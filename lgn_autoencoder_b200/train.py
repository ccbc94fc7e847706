"""The training step of utils/train.py:283-327 (the reference's hot loop body) on the fused path, plus the
data-parallel gradient exchange (SURVEY.md section 8(e)): jets are independent, so the batch is sharded over ranks
with no data-path collective; the only exchange is one NCCL all-reduce(SUM) of the flat gradient per model.

Two entry points:

* ``training_step`` -- the step written with the module API (``LGNEncoder`` / ``LGNDecoder`` forward + autograd), what a
  caller of the reference's ``lgn/`` modules gets unchanged;
* ``FusedTrainStep`` -- the same arithmetic as ONE launch sequence of the C library on static buffers (no autograd
  graph, no per-step allocation), captured in a CUDA graph: normalize -> encoder -> decoder -> chamfer (+ gradient) ->
  decoder adjoint -> encoder adjoint -> L1.  The parameter gradients land in one flat fp64 buffer per model of which
  every ``param.grad`` is a view, so optimizers work unchanged and the all-reduce needs no packing.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
import torch.distributed as dist

from . import _lib, fused
from ._lib import check, ptr


def training_step(encoder, decoder, p4, labels=None, l1_lambda: float = 1e-8, normalize: bool = True, l1_scale: float = 1.0,
                  get_real: str = "real"):
    """normalize_p4('overall_max') -> encoder -> decoder -> get_real(method) + ChamferLoss (sum over the batch)
    + l1_lambda * (|theta_enc|_1 + |theta_dec|_1).  Returns (loss, reconstruction (2,B,N,4), normalised input)."""
    if normalize:
        p4, _ = fused.normalize_p4(p4)
    batch = {"p4": p4}
    if labels is not None:
        batch["labels"] = labels
    latent = encoder(batch, covariance_test=False)
    recon = decoder(latent, covariance_test=False)
    loss = fused.chamfer_loss(recon, p4, get_real)
    if l1_lambda:
        loss = loss + (l1_lambda * l1_scale) * (encoder.l1_norm() + decoder.l1_norm())
    return loss, recon, p4


def allreduce_gradients(*models, group=None):
    """SUM-all-reduce the gradients of every model as one flat fp64 bucket each (chamfer is a sum over jets, so no
    division by the world size; scale the L1 term by 1/world on every rank instead -- ``l1_scale`` above)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    for model in models:
        grads = [p.grad for p in model.parameters() if p.grad is not None]
        if not grads:
            continue
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        off = 0
        for g in grads:
            n = g.numel()
            g.copy_(flat[off:off + n].view_as(g))
            off += n


class FusedTrainStep:
    """One LGAE training step (forward + loss + full backward) for a fixed batch size, on static device buffers.

    ``step(p4, labels=None)`` copies the jets into the static input buffer (host or device source), runs the step and
    returns the loss as a 0-d device tensor; afterwards ``param.grad`` of every encoder / decoder parameter holds the
    gradient of  chamfer_sum + l1_lambda * l1_scale * |theta|_1  (summed over ranks if a process group is active).
    ``recon`` (2,B,N,4), ``latent00/11``, ``norm_factor`` (B,) expose the step's other results.

    ``adjoint`` picks the backward kernels: ``"per_lane"`` (one particle per lane, at most 32 particles per jet) or ``"tiled"``
    (blocks of 32 particles, any particle count, e.g. padded 150-particle jets; ``lgae_train_step_tiled``).  The tiled step
    keeps the encoder's dL/dR of one level in its scratch: B * ceil(N/32) * N * C * 128 doubles, 1.57 GB at B = 512, N = 150,
    C = 4, on top of the workspaces.
    """

    ADJOINTS = ("per_lane", "tiled")

    def __init__(self, encoder, decoder, batch: int, l1_lambda: float = 1e-8, l1_scale: float = 1.0, normalize: bool = True,
                 use_labels: bool = False, use_graph: bool = True, group=None, get_real: str = "real", overlap_allreduce: bool = False,
                 peer_allreduce: bool = False, adjoint: str = "per_lane"):
        if adjoint not in self.ADJOINTS:
            raise ValueError(f"adjoint must be one of {self.ADJOINTS}, not {adjoint!r}")
        if not (getattr(encoder, "fused", False) and getattr(decoder, "fused", False)):
            raise NotImplementedError("FusedTrainStep needs the fused (maxdim 2) encoder and decoder")
        self.enc, self.dec, self.B = encoder, decoder, int(batch)
        self.pe, self.pd = encoder._plan, decoder._plan
        self.tiled = adjoint == "tiled"
        if self.pe.n_particles > 32 and not self.tiled:
            raise NotImplementedError("the per-lane adjoint holds one particle per lane: at most 32 particles per jet "
                                      "(adjoint='tiled' takes any number)")
        self.l1 = float(l1_lambda) * float(l1_scale)
        self.normalize = normalize
        self.get_real = fused.get_real_mode(get_real)
        self.overlap_allreduce = overlap_allreduce
        self.group = group
        self.lib = _lib.load()
        if self.tiled:
            n_part = self.lib.lgae_train_step_tiled_scratch_doubles(C.byref(self.pe.desc), C.byref(self.pd.desc), self.B)
            if n_part == -2:
                reason = self.pe.tiled_reason() or self.pd.tiled_reason() or "a glue kernel of the step does not fit its shared memory"
                raise NotImplementedError(f"configuration not supported by the tiled training step: {reason}")
            if n_part < 0:
                raise ValueError("encoder and decoder do not form one training step (latent widths or particle counts differ)")
        else:
            n_part = self.lib.lgae_train_step_partials_doubles(C.byref(self.pe.desc), C.byref(self.pd.desc), self.B)
        dev = next(encoder.parameters()).device
        self.dev = dev
        f64 = dict(dtype=torch.float64, device=dev)
        B, N = self.B, self.pe.n_particles
        ts, tv = self.pe.latent_taus()
        self.p4_in = torch.zeros((B, N, 4), **f64)
        self.p4 = torch.empty((B, N, 4), **f64) if normalize else self.p4_in
        self.norm_factor = torch.ones(B, **f64)
        self.mask = torch.ones((B, N), dtype=torch.uint8, device=dev) if use_labels else None
        self.ws_e, self.ws_d = self.pe.workspace(B, dev), self.pd.workspace(B, dev)
        self.part = torch.empty(max(int(n_part), 1), **f64)   # partials, or the tiled step's scratch
        self.latent00 = torch.empty((2, B, 1, ts, 1), **f64)
        self.latent11 = torch.empty((2, B, 1, tv, 4), **f64)
        self.sel = torch.empty((4, 2, B, max(self.pe.tau_s, self.pe.tau_v)), dtype=torch.int32, device=dev)
        self.recon = torch.empty((2, B, N, 4), **f64)
        self.g_recon = torch.empty((2, B, N, 4), **f64)
        self.g_lat11 = torch.empty_like(self.latent11)
        self.jet_loss = torch.empty(B, **f64)
        self.loss = torch.zeros((), **f64)
        # one flat gradient bucket for both models (a single all-reduce per step); every param.grad is a view of it
        off_d = (self.pe.n_params + 3) // 4 * 4   # keep the decoder bucket 32-byte aligned
        self.off_d = off_d
        self.g_all = torch.zeros(off_d + self.pd.n_params, **f64)
        # data parallel, opt-in (peer_allreduce=True or LGAE_PEER_ALLREDUCE=1; NCCL's all-reduce is the default, see DESIGN.md
        # section 5 for the measurements): the step's reduce kernels write the local gradient into a bucket that is mapped into
        # every rank of the node (symmetric memory) and one kernel of the library exchanges it over NVLink / NVSwitch
        # (lgae_peer_allreduce: through the switch's multicast object when there is one -- then in place, g_all IS the
        # symmetric bucket --, else by pulling all peers' buckets into g_all)
        self.g_step = self.g_all
        self._peer = None
        import os
        if (peer_allreduce or os.environ.get("LGAE_PEER_ALLREDUCE") == "1") and self._distributed():
            self._setup_peer()
        self.g_e = self.g_all[:self.pe.n_params]
        self.g_d = self.g_all[off_d:]
        self.optimizer = None
        self._probe = (next(encoder.parameters()), next(decoder.parameters()))
        self._bind_grads()
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.use_graph = use_graph
        self._thetas = None
        # pinned host staging: with `step_host` the host->device copy of the jets and the device->host copy of the loss are
        # nodes of the same CUDA graph, so an end-to-end step is one graph launch + one stream synchronisation
        self.host_p4 = torch.zeros((B, N, 4), dtype=torch.float64).pin_memory()
        self.host_mask = torch.ones((B, N), dtype=torch.uint8).pin_memory() if use_labels else None
        self.host_loss = torch.zeros((), dtype=torch.float64).pin_memory()
        self.graph_host: Optional[torch.cuda.CUDAGraph] = None

    def _bind_grads(self):
        for model, plan, flat in ((self.enc, self.pe, self.g_e), (self.dec, self.pd, self.g_d)):
            views = plan.views(flat)
            for name, p in model.named_parameters():
                p.grad = views[name]

    def _setup_peer(self):
        """Collective over the group: allocate the symmetric gradient bucket and exchange the peer mappings."""
        import os
        ok = 0
        state = None
        if True:
            try:
                import torch.distributed._symmetric_memory as symm_mem
                need = int(self.lib.lgae_peer_signal_bytes())
                if symm_mem.get_signal_pad_size() < need:
                    symm_mem.set_signal_pad_size(need)
                g_sym = symm_mem.empty(self.g_all.numel(), dtype=torch.float64, device=self.dev)
                g_sym.zero_()
                hdl = symm_mem.rendezvous(g_sym, self.group if self.group is not None else dist.group.WORLD)
                world = int(hdl.world_size)
                bufs = (C.c_void_p * world)(*[int(p) for p in hdl.buffer_ptrs])
                sigs = (C.c_void_p * world)(*[int(p) for p in hdl.signal_pad_ptrs])
                mc = int(getattr(hdl, "multicast_ptr", 0) or 0) if os.environ.get("LGAE_PEER_MULTICAST", "1") != "0" else 0
                state = (g_sym, hdl, bufs, sigs, int(hdl.rank), world, torch.zeros(1, dtype=torch.int32, device=self.dev), mc)
                ok = 1 if world <= 16 else 0
            except Exception as e:   # noqa: BLE001  (no NVLink peer access, older torch, ...): NCCL carries the exchange
                import logging
                logging.warning(f"lgn_autoencoder_b200: peer-memory all-reduce unavailable ({e!r}); using NCCL")
        flag = torch.tensor([ok], dtype=torch.int32, device=self.dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)     # every rank takes the same path
        has_mc = torch.tensor([1 if (state is not None and state[7]) else 0], dtype=torch.int32, device=self.dev)
        dist.all_reduce(has_mc, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 1:
            if not int(has_mc.item()):
                state = state[:7] + (0,)
            self._peer = state
            self.g_step = state[0]
            if state[7]:
                self.g_all = state[0]     # multicast path: the exchange is in place

    def peer_error(self) -> bool:
        """True if a hand-shake of the peer all-reduce ever timed out on this rank (results are then invalid)."""
        return self._peer is not None and bool(self._peer[6].item())

    def _distributed(self) -> bool:
        return dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1

    def _split(self) -> bool:
        """Two gradient buckets: the decoder's is all-reduced on the library's auxiliary stream while the encoder adjoint runs."""
        return self._distributed() and self._peer is None and self.overlap_allreduce and bool(self.lib.lgae_aux_stream())

    def _phases(self, call):
        """Run ``call(phase)`` as one step (phase 0) or -- data parallel -- as two phases with the all-reduce of the decoder's
        bucket enqueued between them on the auxiliary stream (include/lgae_b200.h: lgae_aux_stream)."""
        if not self._split():
            call(0)
            return
        call(1)
        aux = torch.cuda.ExternalStream(int(self.lib.lgae_aux_stream()), device=self.dev)
        with torch.cuda.stream(aux):
            dist.all_reduce(self.g_d, op=dist.ReduceOp.SUM, group=self.group)
        call(2)

    def _launch(self):
        lib, pe, pd, B = self.lib, self.pe, self.pd, self.B
        st = torch.cuda.current_stream().cuda_stream
        th_e, _ = self.enc._flat_params()
        th_d, _ = self.dec._flat_params()
        self._thetas = (th_e.data_ptr(), th_d.data_ptr())
        fn = lib.lgae_train_step_tiled if self.tiled else lib.lgae_train_step
        self._phases(lambda phase: check(fn(
            C.byref(pe.desc), C.byref(pd.desc), ptr(th_e), ptr(th_d), ptr(self.p4_in), ptr(self.mask), B, 1 if self.normalize else 0,
            ptr(self.p4), ptr(self.norm_factor), ptr(self.ws_e), ptr(self.ws_d), ptr(self.latent00), ptr(self.latent11), ptr(self.sel),
            ptr(self.recon), ptr(self.g_recon), ptr(self.g_lat11), ptr(self.jet_loss), ptr(self.loss), ptr(self.g_step), self.off_d,
            ptr(self.part), self.l1, self.get_real, phase, st), "train_step"))
        self._launch_tail()

    def _launch_tail(self):
        """After the step's kernels: the data-parallel gradient exchange, then the attached optimizer."""
        if self._peer is not None:
            # one kernel: hand-shake with the peers, pull every rank's bucket over NVLink, add in rank order into g_all
            g_sym, _, bufs, sigs, rank, world, err, mc = self._peer
            check(self.lib.lgae_peer_allreduce(bufs, sigs, rank, world, self.g_all.numel(), ptr(self.g_all), mc or None, ptr(err),
                                               torch.cuda.current_stream().cuda_stream), "peer_allreduce")
        elif self._distributed():
            # chamfer is a SUM over jets: all-reduce with SUM, no division by the world size (SURVEY.md section 8(e)); in the
            # split step the decoder's bucket is already being exchanged next to the encoder adjoint
            dist.all_reduce(self.g_e if self._split() else self.g_all, op=dist.ReduceOp.SUM, group=self.group)
        if self.optimizer is not None:
            self.optimizer.step()

    def attach_optimizer(self, optimizer):
        """Make ``optimizer.step()`` (a ``FlatAdam``) the last node of the step: gradients -> (all-reduce) -> parameter update in
        one launch sequence / one CUDA graph.  ``None`` detaches."""
        self.optimizer = optimizer
        self.graph = None
        self.graph_host = None

    def _params_moved(self) -> bool:
        """Cheap per-step check (a few attribute reads): the flat buffers the captured kernels read are still the models'.
        In-place updates (optimizer steps, load_state_dict) keep them; after ``model.to(...)`` or a manual ``param.data = ...``
        call ``refresh()``."""
        te, td = self.enc._theta, self.dec._theta
        return te is None or td is None or self._thetas != (te.data_ptr(), td.data_ptr())

    def refresh(self):
        """Re-validate the parameter aliasing (full check) and drop the captured graphs so that the next step re-captures."""
        self.enc._flat_params()
        self.dec._flat_params()
        self.graph = None
        self.graph_host = None
        self._bind_grads()

    def load(self, p4, labels=None):
        """Copy one batch of jets (host or device tensor, (B,N,4)) into the static input buffer."""
        self.p4_in.copy_(p4, non_blocking=True)
        if self.mask is not None:
            # without labels the reference masks on p4[..., 0] != 0 (lgn_encoder.py:396-398)
            src = labels if labels is not None else p4[..., 0]
            self.mask.copy_((src != 0).to(torch.uint8), non_blocking=True)

    def _check_grads(self):
        """optimizer.zero_grad() (set_to_none=True is torch's default) drops ``param.grad``: point them at the bucket again,
        otherwise optimizer.step() would silently skip every parameter.  O(1): looks at one parameter per model."""
        if self._probe[0].grad is None or self._probe[1].grad is None:
            self._bind_grads()

    def run(self):
        """Run the step on the jets already in the static input buffer."""
        self._check_grads()
        if not self.use_graph:
            self._launch()
            return self.loss
        if self.graph is None or self._params_moved():
            # warm-up on a side stream (caches kernel attributes, NCCL communicators), then capture
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                opt, self.optimizer = self.optimizer, None   # the warm-up run must not update the parameters
                try:
                    self._launch()
                finally:
                    self.optimizer = opt
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._launch()
            self._bind_grads()
        self.graph.replay()
        return self.loss

    def step(self, p4, labels=None):
        self.load(p4, labels)
        return self.run()

    def _launch_host(self):
        """One C call: H2D copy of the pinned jets (+ mask), the step, D2H copy of the loss (``lgae_train_step_host``)."""
        lib, pe, pd, B = self.lib, self.pe, self.pd, self.B
        st = torch.cuda.current_stream().cuda_stream
        th_e, _ = self.enc._flat_params()
        th_d, _ = self.dec._flat_params()
        self._thetas = (th_e.data_ptr(), th_d.data_ptr())
        fn = lib.lgae_train_step_tiled_host if self.tiled else lib.lgae_train_step_host
        self._phases(lambda phase: check(fn(
            C.byref(pe.desc), C.byref(pd.desc), ptr(th_e), ptr(th_d), ptr(self.host_p4), ptr(self.host_mask), ptr(self.host_loss),
            ptr(self.p4_in), ptr(self.mask), B, 1 if self.normalize else 0, ptr(self.p4), ptr(self.norm_factor), ptr(self.ws_e),
            ptr(self.ws_d), ptr(self.latent00), ptr(self.latent11), ptr(self.sel), ptr(self.recon), ptr(self.g_recon), ptr(self.g_lat11),
            ptr(self.jet_loss), ptr(self.loss), ptr(self.g_step), self.off_d, ptr(self.part), self.l1, self.get_real, phase, st),
            "train_step_host"))
        self._launch_tail()

    def step_host(self, p4=None, labels=None) -> float:
        """End-to-end step from host memory: jets (B,N,4) are staged in the pinned buffer ``host_p4`` (pass ``p4=None`` if the
        data loader already wrote them there), copied to the device, the step runs, and the loss comes back as a float."""
        self._check_grads()
        if p4 is not None and p4.data_ptr() != self.host_p4.data_ptr():
            self.host_p4.copy_(p4)
        if self.host_mask is not None and (labels is not None or p4 is not None):
            self.host_mask.copy_(((labels if labels is not None else p4[..., 0]) != 0).to(torch.uint8))
        if not self.use_graph:
            self._launch_host()
        else:
            if self.graph_host is None or self._params_moved():
                s = torch.cuda.Stream()
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    opt, self.optimizer = self.optimizer, None   # the warm-up run must not update the parameters
                    try:
                        self._launch_host()
                    finally:
                        self.optimizer = opt
                torch.cuda.current_stream().wait_stream(s)
                torch.cuda.synchronize()
                self.graph_host = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph_host):
                    self._launch_host()
                self._bind_grads()
            self.graph_host.replay()
        torch.cuda.current_stream().synchronize()
        return float(self.host_loss)


class FlatAdam:
    """``torch.optim.Adam`` (amsgrad=False) for the two models of a ``FusedTrainStep`` as ONE kernel launch per step
    (``lgae_adam_step``) on the flat parameter buffers and the step's flat gradient bucket, instead of two optimizers looping
    over ~130 tensors each (reference: utils/initialize.py:152-158, utils/train.py:342-343).  The step count lives on the
    device, so ``step()`` may be captured in a CUDA graph together with the training step.

    State (``exp_avg``, ``exp_avg_sq`` per model, flat) is exposed through ``state_dict()`` / ``load_state_dict()``."""

    def __init__(self, step: "FusedTrainStep", lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0):
        if lr < 0 or not 0 <= betas[0] < 1 or not 0 <= betas[1] < 1 or eps < 0:
            raise ValueError("invalid Adam hyper-parameters")
        self.fs, self.lr, self.betas, self.eps, self.weight_decay = step, float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        dev = step.dev
        self.exp_avg = [torch.zeros(step.pe.n_params, dtype=torch.float64, device=dev), torch.zeros(step.pd.n_params, dtype=torch.float64, device=dev)]
        self.exp_avg_sq = [torch.zeros_like(self.exp_avg[0]), torch.zeros_like(self.exp_avg[1])]
        self.step_state = torch.zeros(2, dtype=torch.int64, device=dev)   # [updates done, launch counter]
        self.lib = _lib.load()

    def step(self):
        fs = self.fs
        th_e, th_d = fs.enc._theta, fs.dec._theta
        if th_e is None or th_d is None or fs._params_moved():   # cheap pointer check; full re-validation only when needed
            th_e, _ = fs.enc._flat_params()
            th_d, _ = fs.dec._flat_params()
        check(self.lib.lgae_adam_step(ptr(th_e), ptr(fs.g_e), ptr(self.exp_avg[0]), ptr(self.exp_avg_sq[0]), fs.pe.n_params,
                                      ptr(th_d), ptr(fs.g_d), ptr(self.exp_avg[1]), ptr(self.exp_avg_sq[1]), fs.pd.n_params,
                                      self.lr, self.betas[0], self.betas[1], self.eps, self.weight_decay, ptr(self.step_state),
                                      torch.cuda.current_stream().cuda_stream), "adam_step")

    def zero_grad(self, set_to_none: bool = False):
        """No-op: the training step overwrites the gradient bucket."""

    def state_dict(self):
        return {"step": int(self.step_state[0].item()), "exp_avg": [t.clone() for t in self.exp_avg], "exp_avg_sq": [t.clone() for t in self.exp_avg_sq],
                "lr": self.lr, "betas": self.betas, "eps": self.eps, "weight_decay": self.weight_decay}

    def load_state_dict(self, sd):
        self.step_state[0] = int(sd["step"])
        for dst, src in zip(self.exp_avg + self.exp_avg_sq, list(sd["exp_avg"]) + list(sd["exp_avg_sq"])):
            dst.copy_(src)
        self.lr, self.betas, self.eps, self.weight_decay = float(sd["lr"]), tuple(sd["betas"]), float(sd["eps"]), float(sd["weight_decay"])


class FlatRMSprop:
    """``torch.optim.RMSprop`` (centered=False) for both models of a ``FusedTrainStep`` as one launch per step
    (``lgae_rmsprop_step``); the reference builds it with ``eps = get_eps(dtype)`` and ``momentum = 0.9``
    (utils/initialize.py:159-165)."""

    def __init__(self, step: "FusedTrainStep", lr: float = 1e-2, alpha: float = 0.99, eps: float = 1e-8, weight_decay: float = 0.0,
                 momentum: float = 0.0):
        if lr < 0 or alpha < 0 or eps < 0 or momentum < 0:
            raise ValueError("invalid RMSprop hyper-parameters")
        self.fs, self.lr, self.alpha, self.eps, self.weight_decay, self.momentum = step, float(lr), float(alpha), float(eps), float(weight_decay), float(momentum)
        dev = step.dev
        self.square_avg = [torch.zeros(step.pe.n_params, dtype=torch.float64, device=dev), torch.zeros(step.pd.n_params, dtype=torch.float64, device=dev)]
        self.momentum_buf = [torch.zeros_like(t) for t in self.square_avg] if momentum > 0 else [None, None]
        self.lib = _lib.load()

    def step(self):
        fs = self.fs
        th_e, th_d = fs.enc._theta, fs.dec._theta
        if th_e is None or th_d is None or fs._params_moved():
            th_e, _ = fs.enc._flat_params()
            th_d, _ = fs.dec._flat_params()
        check(self.lib.lgae_rmsprop_step(ptr(th_e), ptr(fs.g_e), ptr(self.square_avg[0]), ptr(self.momentum_buf[0]), fs.pe.n_params,
                                         ptr(th_d), ptr(fs.g_d), ptr(self.square_avg[1]), ptr(self.momentum_buf[1]), fs.pd.n_params,
                                         self.lr, self.alpha, self.eps, self.momentum, self.weight_decay,
                                         torch.cuda.current_stream().cuda_stream), "rmsprop_step")

    def zero_grad(self, set_to_none: bool = False):
        """No-op: the training step overwrites the gradient bucket."""


class FusedInference:
    """Forward-only pass (encoder -> decoder -> per-jet chamfer score) for a fixed batch size on static buffers, replayed as one
    CUDA graph: the inference / anomaly-scoring path (test.py:57-95, utils/jet_analysis/anomaly_detection.py chamfer score).
    Jets are independent, so multi-GPU inference is one instance per rank on its shard of the jets, with no communication.
    Supports any number of particles per jet the forward kernels do (blocks of 32 particles per CTA; cfg-5 has 150).

    ``score(p4, labels=None)`` returns the (B,) per-jet chamfer distances between the reconstruction (re + im) and the
    normalised input; ``recon`` (2,B,N,4), ``latent00`` / ``latent11`` and ``norm_factor`` hold the other results.
    """

    def __init__(self, encoder, decoder, batch: int, normalize: bool = True, use_labels: bool = False, use_graph: bool = True,
                 get_real: str = "real"):
        if not (getattr(encoder, "fused_forward", False) and getattr(decoder, "fused_forward", False)):
            raise NotImplementedError("FusedInference needs the fused (maxdim 2 or 3) encoder and decoder")
        self.get_real = fused.get_real_mode(get_real)
        self.enc, self.dec, self.B = encoder, decoder, int(batch)
        self.pe, self.pd = encoder._plan, decoder._plan
        self.normalize = normalize
        self.lib = _lib.load()
        dev = next(encoder.parameters()).device
        f64 = dict(dtype=torch.float64, device=dev)
        B, N = self.B, self.pe.n_particles
        ts, tv = self.pe.latent_taus()
        self.p4_in = torch.zeros((B, N, 4), **f64)
        self.p4 = torch.empty((B, N, 4), **f64) if normalize else self.p4_in
        self.norm_factor = torch.ones(B, **f64)
        self.mask = torch.ones((B, N), dtype=torch.uint8, device=dev) if use_labels else None
        self.ws_e, self.ws_d = self.pe.workspace(B, dev), self.pd.workspace(B, dev)
        self.latent00 = torch.empty((2, B, 1, ts, 1), **f64)
        self.latent11 = torch.empty((2, B, 1, tv, 4), **f64)
        self.sel = torch.empty((4, 2, B, max(self.pe.tau_s, self.pe.tau_v)), dtype=torch.int32, device=dev)
        self.recon = torch.empty((2, B, self.pd.n_particles, 4), **f64)
        self.scores = torch.empty(B, **f64)
        self.use_graph = use_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self._thetas = None

    def _launch(self):
        lib, pe, pd, B = self.lib, self.pe, self.pd, self.B
        st = torch.cuda.current_stream().cuda_stream
        th_e, _ = self.enc._flat_params()
        th_d, _ = self.dec._flat_params()
        self._thetas = (th_e.data_ptr(), th_d.data_ptr())
        if self.normalize:
            check(lib.lgae_normalize_p4(ptr(self.p4_in), B, pe.n_particles, ptr(self.p4), ptr(self.norm_factor), st), "normalize_p4")
        check(lib.lgae_encoder_forward(C.byref(pe.desc), ptr(th_e), ptr(self.p4), ptr(self.mask), B, ptr(self.ws_e), ptr(self.latent00),
                                       ptr(self.latent11), ptr(self.sel), st), "encoder_forward")
        check(lib.lgae_decoder_forward(C.byref(pd.desc), ptr(th_d), ptr(self.latent11), B, ptr(self.ws_d), ptr(self.recon), None, st),
              "decoder_forward")
        check(lib.lgae_chamfer(ptr(self.recon), ptr(self.p4), B, pd.n_particles, pe.n_particles, self.get_real, None, ptr(self.scores), None, None, st),
              "chamfer")

    def all_scores(self, unnormalized: bool = False):
        """After ``score`` / ``run``: every per-jet score of the Cartesian family (``fused.SCORE_NAMES``: chamfer / MSE with the
        Euclidean and the Minkowski metric, jet-level MSEs; utils/jet_analysis/anomaly_detection.py:251-419) of the last batch,
        on the normalised jets or -- ``unnormalized`` -- rescaled by the per-jet normalisation factors as test.py does."""
        return fused.anomaly_scores(self.recon, self.p4, ("real", "imag", "sum", "mean", "norm")[self.get_real],
                                    self.norm_factor if unnormalized else None)

    def run(self):
        if not self.use_graph:
            self._launch()
            return self.scores
        te, td = self.enc._theta, self.dec._theta
        moved = te is None or td is None or self._thetas != (te.data_ptr(), td.data_ptr())
        if self.graph is None or moved:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._launch()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._launch()
        self.graph.replay()
        return self.scores

    def score(self, p4, labels=None):
        self.p4_in.copy_(p4, non_blocking=True)
        if self.mask is not None:
            src = labels if labels is not None else p4[..., 0]
            self.mask.copy_((src != 0).to(torch.uint8), non_blocking=True)
        return self.run()
