"""The one-call training step with the tiled adjoints (FusedTrainStep(adjoint="tiled"), lgae_train_step_tiled): jets of any
particle count as one CUDA graph, against the CPU oracle (oracle/lgae_oracle.py), against the per-lane step at N <= 32, against
the module API at 150 particles, past the persistent grid, with FlatAdam in the graph, and run to run.

Acceptance, as in tests/test_edge_cases_gpu.py: latent, reconstruction and loss within 1e-10 relative of the oracle; every
parameter gradient within 1e-10 * max(|ref|, 1e-4 * gmax)."""
import ctypes as C

import pytest
import torch

from tests.helpers import rel_err
from tests.test_fused_coverage_gpu import TRAIN_CASES, _assert_forward, _assert_grads, _build, _jets
from tests.test_tiled_adjoint_gpu import CAP_CASE, CAP_EXTRA, TILED_CASES, _enc_plan, _oracle_step


@pytest.fixture
def fused_only(monkeypatch):
    """The modules' layer-level composite raises: whatever runs, runs on the fused kernels."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder

    def composite(*args, **kwargs):
        raise AssertionError("the layer-level composite ran")

    monkeypatch.setattr(LGNEncoder, "_forward_generic", composite)
    monkeypatch.setattr(LGNDecoder, "_forward_generic", composite)


def _dec_plan(n, tau_v, channels=(4, 4, 3, 3)):
    from lgn_autoencoder_b200.models import LGNDecoder
    return LGNDecoder(tau_latent_scalars=1, tau_latent_vectors=tau_v, num_output_particles=n, tau_output_scalars=1, tau_output_vectors=1,
                      num_channels=list(channels), maxdim=[2], num_basis_fn=10, max_zf=[1], weight_init="randn", level_gain=[1.0],
                      activation="leakyrelu", mlp=True, mlp_depth=1, mlp_width=1, device=torch.device("cpu"), dtype=torch.float64)


def _models_with_scale(cfg, dev, scale):
    """_build's models, with the encoder's input scale (lgn_encoder.py:371) set to `scale`."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg["seed"])
    common = dict(maxdim=[2], num_basis_fn=cfg["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu",
                  mlp=True, mlp_depth=cfg["mlp_depth"], mlp_width=cfg["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=cfg["tau_s"],
                     tau_latent_vectors=cfg["tau_v"], num_channels=cfg["enc_channels"], jet_features=False,
                     map_to_latent=cfg["map_to_latent"], scale=scale, **common)
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=cfg["tau_s"] * mult, tau_latent_vectors=cfg["tau_v"] * mult, num_output_particles=cfg["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=cfg["dec_channels"], cg_dict=enc.cg_dict, **common)
    assert enc.fused and dec.fused
    return enc.to(dev), dec.to(dev)


def _grads(models):
    return {kind: {k: p.grad.detach().clone() for k, p in m.named_parameters()} for kind, m in models.items()}


def _assert_grads_scaled(name, mine, ref, tol):
    """Every parameter tensor within tol * max(|ref|, 1e-4 * gmax), gmax the largest reference gradient of both models."""
    gmax = max(v.abs().max().item() for part in ref.values() for v in part.values())
    for kind in ref:
        for k, r in ref[kind].items():
            err = (mine[kind][k] - r).abs().max().item()
            assert err <= tol * max(r.abs().max().item(), 1e-4 * gmax), (name, kind, k, err)


def _step_latents(step, cfg):
    lat = {(0, 0): step.latent00, (1, 1): step.latent11}
    if cfg["map_to_latent"] == "sum":   # the module keeps the reference's extra axis of 'sum'
        lat = {k: v.unsqueeze(-3) for k, v in lat.items()}
    return lat


# ---------------------------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_tiled_step_scratch_query_without_gpu():
    """lgae_train_step_tiled_scratch_doubles: -1 for bad arguments, -2 where a tiled adjoint or the fused bridge adjoint does not
    fit its shared memory, otherwise a size that grows with the batch and holds both models' tiled scratch with one shared gA."""
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    enc, dec = _enc_plan(150, [3, 3, 4, 4], "min&max", 1, 8), _dec_plan(150, 16)
    de, dd = C.byref(enc._plan.desc), C.byref(dec._plan.desc)
    q = lib.lgae_train_step_tiled_scratch_doubles
    n1, n8 = q(de, dd, 1), q(de, dd, 8)
    assert 0 < n1 < n8
    for b in (1, 8, 512):
        e, d = lib.lgae_backward_tiled_scratch_doubles(de, b), lib.lgae_backward_tiled_scratch_doubles(dd, b)
        ga_e, ga_d = ((b * 150 * c * 20 + 3) // 4 * 4 for c in (4, 4))
        assert q(de, dd, b) >= e + d - min(ga_e, ga_d), b
    # g_r alone: 1.57 GB at B = 512, N = 150, C = 4
    assert q(de, dd, 512) * 8 > 512 * 5 * 150 * 4 * 128 * 8 > 1.57e9
    # bad arguments
    assert q(de, dd, -1) == -1
    assert q(None, dd, 4) == -1 and q(de, None, 4) == -1
    assert q(dd, de, 4) == -1                                     # decoder and encoder swapped
    assert q(C.byref(_lib.LgaeModelDesc()), dd, 4) == -1
    assert q(de, C.byref(_dec_plan(150, 8)._plan.desc), 4) == -1  # latent widths differ
    assert q(de, C.byref(_dec_plan(140, 16)._plan.desc), 4) == -1  # particle counts differ
    # the 'mix' latent adjoint over 150 x 8 inputs does not fit its shared memory
    mix = _enc_plan(150, [2, 8], "mix", 1, 2)
    assert q(C.byref(mix._plan.desc), C.byref(_dec_plan(150, 2)._plan.desc), 4) == -2
    # each model's tiled adjoint fits on its own, the fused bridge adjoint of the pair does not (8 channels into 8 latent vectors)
    wide = _enc_plan(150, [3, 8], "min&max", 1, 8)
    assert lib.lgae_backward_tiled_scratch_doubles(C.byref(wide._plan.desc), 4) > 0 and lib.lgae_backward_tiled_scratch_doubles(dd, 4) > 0
    assert q(C.byref(wide._plan.desc), dd, 4) == -2
    # the per-lane step's size query is unchanged
    assert lib.lgae_train_step_partials_doubles(de, dd, 8) > 0


def test_tiled_step_refuses_before_any_launch():
    """lgae_train_step_tiled(_host) with a configuration the size query refuses: LGAE_E_UNSUPPORTED without touching the (fake)
    pointers; lgae_train_step still refuses N > 32 the same way."""
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    fake = C.c_void_p(0x1000)
    mix, dec = _enc_plan(150, [2, 8], "mix", 1, 2), _dec_plan(150, 2)
    de, dd = C.byref(mix._plan.desc), C.byref(dec._plan.desc)
    off_d = mix._plan.n_params + 4
    args = [fake] * 3 + [None, 2, 0] + [fake] * 13 + [off_d, fake, 0.0, 0, 0, None]
    assert lib.lgae_train_step_tiled(de, dd, *args) == -2
    assert lib.lgae_train_step(de, dd, *args) == -2
    assert lib.lgae_train_step_tiled_host(de, dd, fake, fake, fake, None, fake, fake, None, 2, 0, *([fake] * 13), off_d, fake, 0.0, 0, 0,
                                          None) == -2


def test_adjoint_argument_without_gpu():
    """An unknown adjoint is a ValueError before anything is allocated; the default still refuses N > 32."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    enc, dec = _enc_plan(40, [3, 3, 4, 4], "min&max", 1, 8), _dec_plan(40, 16)
    with pytest.raises(ValueError, match="adjoint"):
        FusedTrainStep(enc, dec, 2, adjoint="bogus")
    with pytest.raises(NotImplementedError, match="tiled"):
        FusedTrainStep(enc, dec, 2)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TILED_CASES))
def test_tiled_step_matches_oracle(name, fused_only):
    """N = 33-150, every latent map and get_real mode, padded and unpadded: FusedTrainStep(adjoint="tiled") graph-replayed and
    eager against one oracle step (L1 1e-8); the two agree bit for bit."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = TILED_CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, cfg["get_real"], 1e-8)
    p4 = batch_cpu["p4"].to(dev)
    labels = batch_cpu["labels"].to(dev) if cfg["pad"] else None
    results = []
    for use_graph in (True, False):
        step = FusedTrainStep(enc, dec, cfg["batch"], l1_lambda=1e-8, normalize=False, use_labels=cfg["pad"], use_graph=use_graph,
                              get_real=cfg["get_real"], adjoint="tiled")
        for _ in range(2):   # graph: capture, then a replay
            loss = step.step(p4, labels).item()
        torch.cuda.synchronize()
        what = f"{name}/{'graph' if use_graph else 'eager'}"
        _assert_forward(what, _step_latents(step, cfg), step.recon, loss, ref_latent, ref_recon, ref_loss.item())
        _assert_grads(what, models, _grads(models), ref_grads)
        results.append((loss, step.recon.clone(), step.latent11.clone(), step.g_all.clone()))
    (la, ra, za, ga), (lb, rb, zb, gb) = results
    assert la == lb and torch.equal(ra, rb) and torch.equal(za, zb) and torch.equal(ga, gb), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRAIN_CASES))
def test_tiled_step_matches_per_lane_step(name):
    """N <= 32: the tiled step runs the per-lane step's forward, so reconstruction, latents and loss are bit-identical; the
    gradients agree to 1e-12 of each tensor's scale."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = TRAIN_CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    models = {"enc": enc, "dec": dec}
    batch = {k: v.to(dev) for k, v in _jets(cfg, cfg["batch"]).items() if k in ("p4", "labels")}
    out = {}
    for adjoint in ("per_lane", "tiled"):
        step = FusedTrainStep(enc, dec, cfg["batch"], l1_lambda=1e-8, normalize=False, use_labels=cfg["pad"], get_real="sum",
                              adjoint=adjoint)
        for _ in range(2):
            loss = step.step(batch["p4"], batch.get("labels")).item()
        torch.cuda.synchronize()
        out[adjoint] = (loss, step.recon.clone(), step.latent00.clone(), step.latent11.clone(), step.jet_loss.clone(), _grads(models))
    a, b = out["per_lane"], out["tiled"]
    assert a[0] == b[0], (name, a[0], b[0])
    for x, y in zip(a[1:5], b[1:5]):
        assert torch.equal(x, y), name
    _assert_grads_scaled(name, b[5], a[5], 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 2.5])
def test_tiled_step_matches_module_path_at_150_particles(scale, fused_only):
    """cfg-1 at 150 padded particles with normalisation in the step (one CTA per jet normalises and, at input scale 1, runs the
    encoder's input map too): loss, reconstruction and gradients against the module API + autograd (fused forward, tiled
    adjoints as separate calls) within 1e-12."""
    from lgn_autoencoder_b200.train import FusedTrainStep, training_step
    cfg = TILED_CASES["cfg1_n150"]
    dev = torch.device("cuda:0")
    enc, dec = _models_with_scale(cfg, dev, scale)
    models = {"enc": enc, "dec": dec}
    from oracle import lgae_oracle as orc
    raw = orc.synthetic_jets(3, cfg["n"], seed=cfg["seed"] + 3, mass_scale=0.05, pad=True)
    p4, labels = (raw["p4"] * 40.0).to(dev), raw["labels"].to(dev)   # not normalised: the step's first kernel does that
    loss_m, recon_m, _ = training_step(enc, dec, p4, labels=labels, l1_lambda=1e-8, normalize=True, get_real=cfg["get_real"])
    for m in models.values():
        m.zero_grad(set_to_none=True)
    loss_m.backward()
    ref = _grads(models)
    step = FusedTrainStep(enc, dec, 3, l1_lambda=1e-8, normalize=True, use_labels=True, get_real=cfg["get_real"], adjoint="tiled")
    for _ in range(2):
        loss = step.step(p4, labels).item()
    torch.cuda.synchronize()
    assert abs(loss - loss_m.item()) <= 1e-12 * abs(loss_m.item()), (scale, loss, loss_m.item())
    assert rel_err(step.recon, recon_m.detach()) < 1e-12, scale
    _assert_grads_scaled(f"scale {scale}", _grads(models), ref, 1e-12)


@pytest.mark.gpu
def test_tiled_step_replays_split_phases_and_host_entry_are_bit_identical():
    """cfg-1 at 150 particles: two graph replays are bit-identical and equal an eager step; step_host with labels equals step;
    phases 1 + 2 of lgae_train_step_tiled equal phase 0 bit for bit, the decoder's bucket final after phase 1."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200._lib import check, ptr
    from lgn_autoencoder_b200.train import FusedTrainStep
    lib = _lib.load()
    cfg = TILED_CASES["cfg1_n150"]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, 3).items() if k in ("p4", "labels")}
    step = FusedTrainStep(enc, dec, 3, l1_lambda=1e-8, normalize=True, use_labels=True, get_real="sum", adjoint="tiled")
    runs = []
    for _ in range(3):   # capture (+ its warm-up), then two replays
        loss = step.step(batch["p4"], batch["labels"]).item()
        torch.cuda.synchronize()
        runs.append((loss, step.g_all.clone(), step.recon.clone()))
    for l_, g_, r_ in runs[1:]:
        assert l_ == runs[0][0] and torch.equal(g_, runs[0][1]) and torch.equal(r_, runs[0][2])
    l0, g0 = runs[0][0], runs[0][1]
    step.use_graph = False
    assert step.step(batch["p4"], batch["labels"]).item() == l0 and torch.equal(step.g_all, g0)
    step.use_graph = True
    step.mask.zero_()                      # the host entry must upload the mask itself
    assert step.step_host(batch["p4"].cpu(), batch["labels"].cpu()) == l0 and torch.equal(step.g_all, g0)
    assert step.step_host() == l0
    # split step == single call
    step.g_all.zero_()
    assert lib.lgae_aux_stream(), lib.lgae_last_cuda_error()
    pe, pd = step.pe, step.pd
    th_e, _ = enc._flat_params()
    th_d, _ = dec._flat_params()
    st = torch.cuda.current_stream().cuda_stream
    step.load(batch["p4"], batch["labels"])
    for phase in (1, 2):
        check(lib.lgae_train_step_tiled(C.byref(pe.desc), C.byref(pd.desc), ptr(th_e), ptr(th_d), ptr(step.p4_in), ptr(step.mask), step.B, 1,
                                        ptr(step.p4), ptr(step.norm_factor), ptr(step.ws_e), ptr(step.ws_d), ptr(step.latent00),
                                        ptr(step.latent11), ptr(step.sel), ptr(step.recon), ptr(step.g_recon), ptr(step.g_lat11),
                                        ptr(step.jet_loss), ptr(step.loss), ptr(step.g_all), step.off_d, ptr(step.part), step.l1,
                                        step.get_real, phase, st), "train_step_tiled phase")
        if phase == 1:   # the decoder's bucket is final on the auxiliary stream
            aux = torch.cuda.ExternalStream(int(lib.lgae_aux_stream()), device=dev)
            aux.synchronize()
            assert torch.equal(step.g_d, g0[step.off_d:])
    torch.cuda.synchronize()
    assert step.loss.item() == l0 and torch.equal(step.g_all, g0)


@pytest.mark.gpu
def test_tiled_step_batch_past_the_persistent_grid(fused_only):
    """Batch 4 * SMs + 37 at N = 40: the level and glue adjoints walk more units than they have CTAs.  The full batch against
    the same jets in chunks below the cap: reconstruction and per-jet losses bit-identical, gradient sums within 1e-11."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = CAP_CASE
    dev = torch.device("cuda:0")
    sms = int(_lib.load().lgae_device_sm_count())
    B = 4 * sms + CAP_EXTRA
    enc, dec = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, B).items() if k in ("p4", "labels")}
    full = FusedTrainStep(enc, dec, B, l1_lambda=0.0, normalize=False, use_labels=True, get_real="sum", adjoint="tiled")
    for _ in range(2):
        full.step(batch["p4"], batch["labels"])
    torch.cuda.synchronize()
    g_full, recon, jet_loss = full.g_all.clone(), full.recon.clone(), full.jet_loss.clone()
    chunk = 2 * sms - 1   # 2 blocks per jet: fewer than 4 * SMs units
    g_sum = torch.zeros_like(g_full)
    for lo in range(0, B, chunk):
        hi = min(lo + chunk, B)
        part = FusedTrainStep(enc, dec, hi - lo, l1_lambda=0.0, normalize=False, use_labels=True, use_graph=False, get_real="sum",
                              adjoint="tiled")
        part.step(batch["p4"][lo:hi], batch["labels"][lo:hi])
        torch.cuda.synchronize()
        assert torch.equal(part.recon, recon[:, lo:hi]) and torch.equal(part.jet_loss, jet_loss[lo:hi]), lo
        g_sum += part.g_all
    assert (g_sum - g_full).abs().max().item() <= 1e-11 * g_full.abs().max().item()


@pytest.mark.gpu
def test_tiled_step_with_flat_adam_matches_module_path_and_torch_adam(fused_only):
    """cfg-1 at 150 particles: FlatAdam attached to the tiled step (one graph per step) against the module API + two
    torch.optim.Adam on a copy of the models; parameters after 3 steps within 1e-11."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FlatAdam, FusedTrainStep
    cfg = TILED_CASES["cfg1_n150"]
    dev = torch.device("cuda:0")
    enc_a, dec_a = _build(cfg, dev)
    enc_b, dec_b = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, 2).items() if k in ("p4", "labels")}
    lr, wd = 3e-3, 1e-2
    opts = [torch.optim.Adam(enc_a.parameters(), lr, weight_decay=wd), torch.optim.Adam(dec_a.parameters(), lr, weight_decay=wd)]
    step = FusedTrainStep(enc_b, dec_b, 2, l1_lambda=1e-8, normalize=False, use_labels=True, get_real=cfg["get_real"], adjoint="tiled")
    step.attach_optimizer(FlatAdam(step, lr=lr, weight_decay=wd))
    for _ in range(3):
        for o in opts:
            o.zero_grad()
        la = fused.chamfer_loss(dec_a(enc_a(batch)), batch["p4"], cfg["get_real"]) + 1e-8 * (enc_a.l1_norm() + dec_a.l1_norm())
        la.backward()
        for o in opts:
            o.step()
        lb = step.step(batch["p4"], batch["labels"]).item()
        assert abs(la.item() - lb) <= 1e-11 * abs(la.item())
    torch.cuda.synchronize()
    for (k, pa), (_, pb) in zip(list(enc_a.named_parameters()) + list(dec_a.named_parameters()),
                                list(enc_b.named_parameters()) + list(dec_b.named_parameters())):
        assert rel_err(pb, pa) < 1e-11, k
