"""FusedTrainStep (static buffers + CUDA graph) against the module/autograd path and the reference's golden vectors."""
import pytest
import torch

from tests.helpers import assert_grads_close, load_golden, rel_err
from tests.test_models_gpu import load

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("use_graph", [False, True])
def test_fused_train_step_matches_reference(use_graph):
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")
    g, enc, dec, batch = load("cfg1_b3", dev)
    step = FusedTrainStep(enc, dec, batch["p4"].shape[0], l1_lambda=1e-8, normalize=False, use_graph=use_graph, get_real="sum")
    for _ in range(3):   # replays must be idempotent
        loss = step.step(batch["p4"])
    torch.cuda.synchronize()
    assert abs(loss.item() - g["loss"].item()) < 1e-10 * abs(g["loss"].item())
    assert rel_err(step.recon, g["recons"]) < 1e-10
    assert rel_err(step.latent11, g["latent"]["(1, 1)"]) < 1e-10
    assert_grads_close({k: p.grad for k, p in enc.named_parameters()}, g["grads_enc"])
    assert_grads_close({k: p.grad for k, p in dec.named_parameters()}, g["grads_dec"])


def test_fused_train_step_padded_jets_and_optimizer():
    """labels mask, normalisation, and an optimizer step between replays (weights are read from the live buffers)."""
    from lgn_autoencoder_b200.train import FusedTrainStep, training_step
    dev = torch.device("cuda:0")
    g, enc, dec, batch = load("pad_n8", dev)
    b = batch["p4"].shape[0]
    step = FusedTrainStep(enc, dec, b, l1_lambda=1e-8, normalize=True, use_labels=True, use_graph=True, get_real="sum")
    opt = torch.optim.SGD(list(enc.parameters()) + list(dec.parameters()), lr=1e-4)
    l0 = step.step(batch["p4"], batch["labels"]).item()
    # the same step through the module API + autograd
    g_fused = {k: p.grad.clone() for k, p in list(enc.named_parameters()) + list(dec.named_parameters())}
    for p in list(enc.parameters()) + list(dec.parameters()):
        p.grad = None
    loss, _, _ = training_step(enc, dec, batch["p4"], labels=batch["labels"], l1_lambda=1e-8, get_real="sum")
    loss.backward()
    assert abs(loss.item() - l0) < 1e-12 * abs(l0)
    g_mod = {k: p.grad.clone() for k, p in list(enc.named_parameters()) + list(dec.named_parameters())}
    gmax = max(v.abs().max().item() for v in g_mod.values())
    for k in g_mod:
        assert (g_mod[k] - g_fused[k]).abs().max().item() <= 1e-12 * gmax, k
    step._bind_grads()
    l1 = step.step(batch["p4"], batch["labels"]).item()
    assert l1 == l0
    opt.step()
    l2 = step.step(batch["p4"], batch["labels"]).item()
    assert l2 != l0


def test_step_host_matches_step():
    """End-to-end entry (pinned staging + in-graph copies) gives the same loss and gradients as the device-resident step."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")
    g, enc, dec, batch = load("cfg1_b3", dev)
    step = FusedTrainStep(enc, dec, batch["p4"].shape[0], l1_lambda=1e-8, normalize=False, use_graph=True, get_real="sum")
    l_dev = step.step(batch["p4"]).item()
    g_dev = step.g_e.clone()
    for _ in range(2):
        l_host = step.step_host(batch["p4"].cpu())
    assert l_host == l_dev
    assert torch.equal(step.g_e, g_dev)
    assert abs(l_host - g["loss"].item()) < 1e-10 * abs(g["loss"].item())


def test_fused_inference_matches_module_forward_and_oracle_at_150_particles():
    """Forward-only scoring path at the cfg-5 particle count (150 per jet: five particle blocks per CTA in the forward kernels)
    against the module forward and against the CPU oracle on two seeded jets."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedInference
    from oracle import lgae_oracle as orc
    from tests.test_edge_cases_gpu import _build
    dev = torch.device("cuda:0")
    cfg = dict(seed=21, n=150, enc_channels=[3, 3, 4, 4], dec_channels=[4, 4, 3, 3], tau_s=1, tau_v=8, map_to_latent="min&max", mlp_depth=6,
               mlp_width=6)
    enc, dec = _build(cfg, dev)
    data = orc.synthetic_jets(2, 150, seed=22, mass_scale=1e-6, pad=True)
    inf = FusedInference(enc, dec, 2, normalize=True, use_labels=True, get_real="sum")
    for _ in range(2):
        scores = inf.score(data["p4"], data["labels"]).clone()
    # module path
    p4n, _ = fused.normalize_p4(data["p4"].to(dev))
    with torch.no_grad():
        rec = dec(enc({"p4": p4n, "labels": data["labels"].to(dev)}))
    assert torch.equal(rec, inf.recon)
    assert torch.equal(fused.chamfer_per_jet(rec, p4n, "sum"), scores)
    # oracle
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    enc_sd = {k: v.detach().cpu() for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu() for k, v in dec.state_dict().items()}
    with torch.no_grad():
        lat = orc.encoder_forward(enc_sd, dict(num_channels=cfg["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent="min&max"),
                                  dict(data, p4=pn))
        ref = orc.decoder_forward(dec_sd, dict(num_channels=cfg["dec_channels"], maxdim=[2], max_zf=[1]), lat)
    assert rel_err(inf.recon, ref) < 1e-10
    x = orc.get_real_sum(ref)
    for b in range(2):
        s = orc.chamfer_loss(x[b:b + 1], pn[b:b + 1]).item()
        assert abs(scores[b].item() - s) <= 1e-10 * abs(s)


@pytest.mark.parametrize("in_graph", [False, True])
def test_flat_adam_matches_torch_adam(in_graph):
    """FlatAdam (one launch for both models, optionally a node of the step's CUDA graph) follows torch.optim.Adam on the same
    gradients for several steps; a caller's zero_grad(set_to_none=True) does not detach the gradient views."""
    from lgn_autoencoder_b200.train import FlatAdam, FusedTrainStep
    dev = torch.device("cuda:0")
    g, enc_a, dec_a, batch = load("cfg1_b3", dev)
    _, enc_b, dec_b, _ = load("cfg1_b3", dev)
    b = batch["p4"].shape[0]
    lr, wd = 3e-3, 1e-2
    sa = FusedTrainStep(enc_a, dec_a, b, l1_lambda=1e-8, normalize=True, use_graph=True, get_real="sum")
    opts = [torch.optim.Adam(enc_a.parameters(), lr, weight_decay=wd), torch.optim.Adam(dec_a.parameters(), lr, weight_decay=wd)]
    sb = FusedTrainStep(enc_b, dec_b, b, l1_lambda=1e-8, normalize=True, use_graph=True, get_real="sum")
    flat = FlatAdam(sb, lr=lr, weight_decay=wd)
    if in_graph:
        sb.attach_optimizer(flat)
    losses_a, losses_b = [], []
    for it in range(5):
        for o in opts:
            o.zero_grad()                       # set_to_none=True: FusedTrainStep must re-bind its gradient views
        losses_a.append(sa.step(batch["p4"]).item())
        for o in opts:
            o.step()
        losses_b.append(sb.step(batch["p4"]).item())
        if not in_graph:
            flat.step()
    torch.cuda.synchronize()
    assert losses_a[0] == losses_b[0] and losses_a[-1] != losses_a[0]
    for x, y in zip(losses_a, losses_b):
        assert abs(x - y) <= 1e-11 * abs(x)
    assert int(flat.step_state[0].item()) == 5 and int(flat.step_state[1].item()) == 0
    for (k, pa), (_, pb) in zip(list(enc_a.named_parameters()) + list(dec_a.named_parameters()),
                                list(enc_b.named_parameters()) + list(dec_b.named_parameters())):
        assert rel_err(pb, pa) < 1e-11, k
    # optimizer state round trip
    sd = flat.state_dict()
    flat2 = FlatAdam(sb, lr=1.0)
    flat2.load_state_dict(sd)
    assert flat2.lr == lr and int(flat2.step_state[0].item()) == 5 and torch.equal(flat2.exp_avg[1], flat.exp_avg[1])


def test_flat_rmsprop_matches_torch_rmsprop():
    """The reference's other optimizer choice (momentum 0.9) on the flat buffers, one launch for both models."""
    from lgn_autoencoder_b200.train import FlatRMSprop, FusedTrainStep
    dev = torch.device("cuda:0")
    g, enc_a, dec_a, batch = load("cfg1_b3", dev)
    _, enc_b, dec_b, _ = load("cfg1_b3", dev)
    b = batch["p4"].shape[0]
    kw = dict(lr=2e-3, eps=1e-16, momentum=0.9)
    sa = FusedTrainStep(enc_a, dec_a, b, l1_lambda=1e-8, use_graph=True, get_real="sum")
    opts = [torch.optim.RMSprop(enc_a.parameters(), **kw), torch.optim.RMSprop(dec_a.parameters(), **kw)]
    sb = FusedTrainStep(enc_b, dec_b, b, l1_lambda=1e-8, use_graph=True, get_real="sum")
    sb.attach_optimizer(FlatRMSprop(sb, **kw))
    for it in range(4):
        la = sa.step(batch["p4"]).item()
        for o in opts:
            o.step()
        lb = sb.step(batch["p4"]).item()
        assert abs(la - lb) <= 1e-10 * abs(la)
    for (k, pa), (_, pb) in zip(list(enc_a.named_parameters()) + list(dec_a.named_parameters()),
                                list(enc_b.named_parameters()) + list(dec_b.named_parameters())):
        assert rel_err(pb, pa) < 1e-10, k


def test_full_size_step_properties():
    """BASELINE configs[1] at its full size (512 jets x 30 particles per GPU), where the CPU oracle is too slow to be the
    checker: size-independent properties of the path.  (1) Jets are independent and chamfer is a SUM over jets, so the step on
    512 jets equals the two half-batch steps: per-jet reconstructions and losses identical, parameter gradients additive.
    (2) The encoder's min&max pooling and every neighbour sum are permutation invariant: permuting the particles inside each
    jet leaves latent, reconstruction and loss unchanged (up to summation order)."""
    from bench import CFG, build_models, synthetic_jets
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")
    enc, dec = build_models(dev)
    B, N = CFG["batch"], CFG["n"]
    assert (B, N) == (512, 30)
    p4 = synthetic_jets(B, N, seed=11).to(dev)
    full = FusedTrainStep(enc, dec, B, l1_lambda=0.0, use_graph=True, get_real="sum")
    half = FusedTrainStep(enc, dec, B // 2, l1_lambda=0.0, use_graph=False, get_real="sum")
    loss = full.step(p4).item()
    g_full, recon, jet_loss, lat = full.g_all.clone(), full.recon.clone(), full.jet_loss.clone(), full.latent11.clone()
    assert torch.isfinite(g_full).all() and g_full.abs().max().item() > 0
    g_sum, l_sum = torch.zeros_like(g_full), 0.0
    for h in range(2):
        sl = slice(h * B // 2, (h + 1) * B // 2)
        l_sum += half.step(p4[sl]).item()
        g_sum += half.g_all
        assert torch.equal(half.recon, recon[:, sl]) and torch.equal(half.jet_loss, jet_loss[sl])   # per-jet work is batch independent
    assert abs(l_sum - loss) <= 1e-12 * abs(loss)
    assert (g_sum - g_full).abs().max().item() <= 1e-11 * g_full.abs().max().item()
    assert abs(jet_loss.sum().item() - loss) <= 1e-12 * abs(loss)
    # permutation of the particles inside every jet
    gen = torch.Generator().manual_seed(3)
    perm = torch.stack([torch.randperm(N, generator=gen) for _ in range(B)]).to(dev)
    p4p = torch.gather(p4, 1, perm[:, :, None].expand(B, N, 4))
    full._bind_grads()
    loss_p = full.step(p4p).item()
    assert abs(loss_p - loss) <= 1e-10 * abs(loss)
    assert rel_err(full.latent11, lat) < 1e-10 and rel_err(full.recon, recon) < 1e-10
    assert (full.g_all - g_full).abs().max().item() <= 1e-9 * g_full.abs().max().item()


def test_step_host_with_padded_jets_matches_step():
    """lgae_train_step_host also carries the labels mask from pinned host memory."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")
    g, enc, dec, batch = load("pad_n8", dev)
    b = batch["p4"].shape[0]
    step = FusedTrainStep(enc, dec, b, l1_lambda=1e-8, normalize=True, use_labels=True, use_graph=True, get_real="sum")
    l_dev = step.step(batch["p4"], batch["labels"]).item()
    g_dev = step.g_all.clone()
    step.mask.zero_()                      # make sure the host entry really re-uploads the mask
    l_host = step.step_host(batch["p4"].cpu(), batch["labels"].cpu())
    assert l_host == l_dev and torch.equal(step.g_all, g_dev)
    assert l_host == step.step_host()      # replay from the staged pinned buffers


@pytest.mark.parametrize("variant", ["near_massless", "padded_labels"])
def test_cfg1_full_batch_matches_oracle(variant):
    """BASELINE configs[1] at its REAL batch (512 jets x 30 particles) against the CPU oracle on the same weights and jets
    (about 3 s of CPU work per variant): FusedTrainStep (CUDA graph, the benchmarked path) and the module/autograd path --
    latent (0,0) / (1,1), reconstruction, loss and every parameter gradient within 1e-10.  The persistent kernels take a
    different trip count at 15 360 rows than in the 3-jet fixtures."""
    from bench import CFG, build_models
    from lgn_autoencoder_b200.train import FusedTrainStep, training_step
    from oracle import lgae_oracle as orc
    dev = torch.device("cuda:0")
    enc, dec = build_models(dev)
    B, N = CFG["batch"], CFG["n"]
    data = orc.synthetic_jets(B, N, seed=21, mass_scale=1e-6, pad=(variant == "padded_labels"))
    labels = data.get("labels")
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    enc_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in dec.state_dict().items()}
    ecfg = dict(num_channels=CFG["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent=CFG["map_to_latent"])
    dcfg = dict(num_channels=CFG["dec_channels"], maxdim=[2], max_zf=[1])
    batch = {"p4": pn} if labels is None else {"p4": pn, "labels": labels}
    ref_loss, ref_lat, ref_recon = orc.training_step(enc_sd, dec_sd, ecfg, dcfg, batch, l1_lambda=CFG["l1_lambda"])
    ref_loss.backward()
    ref_ge, ref_gd = {k: v.grad for k, v in enc_sd.items()}, {k: v.grad for k, v in dec_sd.items()}

    step = FusedTrainStep(enc, dec, B, l1_lambda=CFG["l1_lambda"], normalize=True, use_labels=labels is not None, use_graph=True,
                          get_real="sum")
    for _ in range(2):
        loss = step.step(data["p4"].to(dev), None if labels is None else labels.to(dev)).item()
    errs = {"loss": abs(loss - ref_loss.item()) / abs(ref_loss.item()), "recon": rel_err(step.recon, ref_recon),
            "lat00": rel_err(step.latent00, ref_lat[(0, 0)]), "lat11": rel_err(step.latent11, ref_lat[(1, 1)])}
    print(variant, "fused step", {k: f"{v:.2e}" for k, v in errs.items()})
    assert all(v < 1e-10 for v in errs.values()), errs
    assert_grads_close({k: p.grad for k, p in enc.named_parameters()}, ref_ge)
    assert_grads_close({k: p.grad for k, p in dec.named_parameters()}, ref_gd)
    # the module API + autograd on the same jets
    for p in list(enc.parameters()) + list(dec.parameters()):
        p.grad = None
    loss_m, recon_m, _ = training_step(enc, dec, data["p4"].to(dev), labels=None if labels is None else labels.to(dev),
                                       l1_lambda=CFG["l1_lambda"], get_real="sum")
    loss_m.backward()
    assert abs(loss_m.item() - ref_loss.item()) < 1e-10 * abs(ref_loss.item())
    assert rel_err(recon_m, ref_recon) < 1e-10
    assert_grads_close({k: p.grad for k, p in enc.named_parameters()}, ref_ge)
    assert_grads_close({k: p.grad for k, p in dec.named_parameters()}, ref_gd)


@pytest.mark.parametrize("name", ["real_n6", "norm_n6"])
def test_fused_train_step_get_real_modes(name):
    """get_real 'real' (the reference's default, main.py:295-300) and 'norm' through the fused step, against the reference."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")
    g, enc, dec, batch = load(name, dev)
    step = FusedTrainStep(enc, dec, batch["p4"].shape[0], l1_lambda=1e-8, normalize=False, get_real=g["cfg"]["get_real"])
    loss = step.step(batch["p4"]).item()
    assert abs(loss - g["loss"].item()) < 1e-10 * abs(g["loss"].item())
    assert rel_err(step.recon, g["recons"]) < 1e-10
    assert_grads_close({k: p.grad for k, p in enc.named_parameters()}, g["grads_enc"])
    assert_grads_close({k: p.grad for k, p in dec.named_parameters()}, g["grads_dec"])


def test_anomaly_scores_match_reference_and_oracle():
    """(f3) lgae_anomaly_scores: chamfer / MSE with the Euclidean and the Minkowski metric and the jet-level scores
    (utils/jet_analysis/anomaly_detection.py:251-419) against the reference's golden values, and through FusedInference against the
    oracle on the model's own reconstruction (normalised and rescaled by the per-jet factors)."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedInference
    from oracle import lgae_oracle as orc
    dev = torch.device("cuda:0")
    g = load_golden("anomaly_scores")
    recon_c = torch.stack([g["recons"], 0.3 * g["recons"]]).to(dev)     # complex (2,B,N,4); 'real' picks the first plane
    mine = fused.anomaly_scores(recon_c, g["target"].to(dev), "real")
    for short, name in (("chamfer_cartesian", "chamfer_particle_cartesian"), ("mse_cartesian", "mse_particle_cartesian"),
                        ("chamfer_lorentz", "chamfer_particle_lorentz"), ("mse_lorentz", "mse_particle_lorentz"),
                        ("jet_cartesian", "jet_cartesian"), ("jet_lorentz", "jet_lorentz")):
        assert rel_err(mine[name], g[short]) < 1e-10, name
    _, enc, dec, batch = load("cfg1_b3", dev)
    inf = FusedInference(enc, dec, batch["p4"].shape[0], normalize=True, get_real="sum")
    p4 = batch["p4"] * 3.7
    inf.score(p4)
    x = (inf.recon[0] + inf.recon[1]).cpu()
    for unnorm in (False, True):
        f = inf.norm_factor.cpu().view(-1, 1, 1) if unnorm else 1.0
        ref = orc.anomaly_scores_cartesian(x * f, inf.p4.cpu() * f)
        got = inf.all_scores(unnormalized=unnorm)
        for name in fused.SCORE_NAMES:
            # the Minkowski scores are differences of squares (near-cancelling for a good reconstruction): their error is
            # measured against the Euclidean counterpart's scale
            scale = ref[name.replace("lorentz", "cartesian")].abs().max().item()
            assert (got[name].cpu() - ref[name]).abs().max().item() < 1e-10 * scale, (name, unnorm)


def test_peer_allreduce_single_rank_and_split_step():
    """lgae_peer_allreduce with world = 1 (the hand-shakes have no peer, the pull is the identity; the multi-rank behaviour is
    checked by tools/dp_check.py under torchrun) and the two-phase form of lgae_train_step (decoder bucket final after phase 1,
    the rest in phase 2 with the auxiliary stream joined back) against the single call."""
    import ctypes as C
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200._lib import check, ptr
    from lgn_autoencoder_b200.train import FusedTrainStep
    lib = _lib.load()
    dev = torch.device("cuda:0")
    n = 1001
    buf = torch.randn(n + 1, dtype=torch.float64, device=dev)[:n]          # odd length, 16-byte aligned start
    out = torch.empty(n + 1, dtype=torch.float64, device=dev)[:n]
    sig = torch.zeros(int(lib.lgae_peer_signal_bytes()) // 4, dtype=torch.int32, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    bufs, sigs = (C.c_void_p * 1)(buf.data_ptr()), (C.c_void_p * 1)(sig.data_ptr())
    st = torch.cuda.current_stream().cuda_stream
    check(lib.lgae_peer_allreduce(bufs, sigs, 0, 1, n, ptr(out), None, ptr(err), st), "peer_allreduce")
    torch.cuda.synchronize()
    assert torch.equal(out, buf) and int(err.item()) == 0 and int(sig.abs().sum().item()) == 0
    assert lib.lgae_peer_allreduce(bufs, sigs, 1, 1, n, ptr(out), None, ptr(err), st) == -1      # rank out of range
    # split step == single call
    g, enc, dec, batch = load("cfg1_b3", dev)
    step = FusedTrainStep(enc, dec, batch["p4"].shape[0], l1_lambda=1e-8, normalize=False, use_graph=False, get_real="sum")
    l0 = step.step(batch["p4"]).item()
    g0 = step.g_all.clone()
    step.g_all.zero_()
    assert lib.lgae_aux_stream(), lib.lgae_last_cuda_error()
    pe, pd = step.pe, step.pd
    th_e, _ = enc._flat_params()
    th_d, _ = dec._flat_params()
    for phase in (1, 2):
        check(lib.lgae_train_step(C.byref(pe.desc), C.byref(pd.desc), ptr(th_e), ptr(th_d), ptr(step.p4_in), ptr(step.mask), step.B, 0,
                                  ptr(step.p4), ptr(step.norm_factor), ptr(step.ws_e), ptr(step.ws_d), ptr(step.latent00), ptr(step.latent11),
                                  ptr(step.sel), ptr(step.recon), ptr(step.g_recon), ptr(step.g_lat11), ptr(step.jet_loss), ptr(step.loss),
                                  ptr(step.g_all), step.off_d, ptr(step.part), step.l1, step.get_real, phase, st), "train_step phase")
        if phase == 1:   # the decoder's bucket is final on the auxiliary stream
            aux = torch.cuda.ExternalStream(int(lib.lgae_aux_stream()), device=dev)
            aux.synchronize()
            assert torch.equal(step.g_d, g0[step.off_d:])
    torch.cuda.synchronize()
    assert step.loss.item() == l0 and torch.equal(step.g_all, g0)
    # phase 2 without phase 1 is refused
    assert lib.lgae_train_step(C.byref(pe.desc), C.byref(pd.desc), ptr(th_e), ptr(th_d), ptr(step.p4_in), ptr(step.mask), step.B, 0,
                               ptr(step.p4), ptr(step.norm_factor), ptr(step.ws_e), ptr(step.ws_d), ptr(step.latent00), ptr(step.latent11),
                               ptr(step.sel), ptr(step.recon), ptr(step.g_recon), ptr(step.g_lat11), ptr(step.jet_loss), ptr(step.loss),
                               ptr(step.g_all), step.off_d, ptr(step.part), step.l1, step.get_real, 2, st) == -1


def test_bench_dump_outputs_are_the_timed_step_results(tmp_path):
    """bench.py --dump-outputs writes the loss, reconstruction, latents, normalisation and gradients of its timed step; they
    match the same step run here on the same seeded models and jets, and --steps is the number of timed steps it reports."""
    import json
    import os
    import subprocess
    import sys

    import numpy as np

    from bench import CFG, build_models, synthetic_jets
    from lgn_autoencoder_b200.train import FusedTrainStep
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    B, out = 16, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0", "--batch", str(B),
                        "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(out)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2
    dev = torch.device("cuda:0")
    enc, dec = build_models(dev)
    step = FusedTrainStep(enc, dec, B, l1_lambda=CFG["l1_lambda"], normalize=True, get_real="sum")
    loss = step.step(synthetic_jets(B, CFG["n"], seed=100).to(dev))
    torch.cuda.synchronize()
    want = {"loss": loss, "recon": step.recon, "latent00": step.latent00, "latent11": step.latent11, "norm_factor": step.norm_factor,
            "grad_encoder": torch.cat([p.grad.reshape(-1) for _, p in enc.named_parameters()]),
            "grad_decoder": torch.cat([p.grad.reshape(-1) for _, p in dec.named_parameters()])}
    assert sorted(os.listdir(out)) == sorted(f"{k}.npy" for k in want)
    for name, ref in want.items():
        got = np.load(out / f"{name}.npy")
        assert got.dtype == np.float64 and got.shape == tuple(ref.shape), name
        assert rel_err(torch.from_numpy(got), ref) < 1e-12, (name, rel_err(torch.from_numpy(got), ref))


def test_bench_dump_outputs_sample_jets_past_the_size_limit(tmp_path, monkeypatch):
    """When the per-jet arrays would take the dump past its size limit, it keeps a seeded, sorted sample of jets: jet_index
    lists them, recon / latents are cut along the batch axis (1) and norm_factor along its only axis, and the files fit."""
    import os

    import numpy as np

    import bench
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")
    B = 16
    enc, dec = bench.build_models(dev)
    step = FusedTrainStep(enc, dec, B, l1_lambda=bench.CFG["l1_lambda"], normalize=True, get_real="sum")
    step.step(bench.synthetic_jets(B, bench.CFG["n"], seed=100).to(dev))
    torch.cuda.synchronize()
    n_grad = sum(p.numel() for m in (enc, dec) for p in m.parameters())
    limit = 8 * (n_grad + 1) + 4096 + 6 * 2560     # room for the gradients, the loss, the headers and a few jets
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    out = tmp_path / "dump"
    bench.dump_outputs(str(out), step)
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= limit
    idx = np.load(out / "jet_index.npy")
    assert idx.dtype == np.float64 and 0 < len(idx) < B and np.all(np.diff(idx) > 0)
    sel = torch.from_numpy(idx.astype(np.int64)).to(dev)
    for name, t, axis in (("recon", step.recon, 1), ("latent00", step.latent00, 1), ("latent11", step.latent11, 1), ("norm_factor", step.norm_factor, 0)):
        assert np.array_equal(np.load(out / f"{name}.npy"), t.index_select(axis, sel).cpu().numpy()), name
    assert np.array_equal(np.load(out / "loss.npy"), step.loss.cpu().numpy())
    bench.dump_outputs(str(tmp_path / "again"), step)
    assert np.array_equal(np.load(tmp_path / "again" / "jet_index.npy"), idx)
