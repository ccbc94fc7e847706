"""GPU parity of the whole-model C entry points against the golden vectors of the unmodified reference and
against the stage-level torch restatement.  Run on the B200 box: pytest -m gpu."""
from collections import OrderedDict

import pytest
import torch

from tests.helpers import assert_grads_close, grad_errors, load_golden, rel_err

pytestmark = pytest.mark.gpu

CASES = ["cfg1_b3", "pad_n8", "mean_n6"]


def _plans(g):
    from lgn_autoencoder_b200.fused import FusedPlan
    cfg = g["cfg"]
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    common = dict(n_particles=cfg["n"], num_basis_fn=10, mlp=True, mlp_depth=cfg.get("mlp_depth", 6), mlp_width=cfg.get("mlp_width", 6))
    enc = FusedPlan("encoder", OrderedDict((k, tuple(v.shape)) for k, v in g["enc_state"].items()), channels=cfg["enc_channels"],
                    latent_mode=cfg["map_to_latent"], tau_s=cfg["tau_s"], tau_v=cfg["tau_v"], **common)
    dec = FusedPlan("decoder", OrderedDict((k, tuple(v.shape)) for k, v in g["dec_state"].items()), channels=cfg["dec_channels"],
                    tau_s=cfg["tau_s"] * mult, tau_v=cfg["tau_v"] * mult, **common)
    return enc, dec


def _run(g, dev):
    from lgn_autoencoder_b200 import fused
    enc, dec = _plans(g)
    th_e = enc.flatten(g["enc_state"], dev)
    th_d = dec.flatten(g["dec_state"], dev)
    p4 = g["batch"]["p4"].to(dev).contiguous()
    mask = None
    if "labels" in g["batch"]:
        mask = (g["batch"]["labels"] != 0).to(torch.uint8).to(dev).contiguous()
    lat00, lat11, ws_e, sel = fused.encoder_forward_raw(enc, th_e, p4, mask)
    recon, gen00, ws_d = fused.decoder_forward_raw(dec, th_d, lat11, want_gen00=True)
    return dict(enc=enc, dec=dec, th_e=th_e, th_d=th_d, p4=p4, mask=mask, lat00=lat00, lat11=lat11, ws_e=ws_e, sel=sel,
                recon=recon, gen00=gen00, ws_d=ws_d)


@pytest.mark.parametrize("name", CASES + ["n40_b2"])
def test_forward_matches_reference(name):
    dev = torch.device("cuda:0")
    g = load_golden(name)
    r = _run(g, dev)
    torch.cuda.synchronize()
    errs = {}
    # every internal GVec the reference exposes with covariance_test=True
    b = r["p4"].shape[0]
    ne = r["enc"].n_levels
    mine_nodes = [r["enc"].node_features(r["ws_e"], b, l) for l in range(ne + 1)]
    mine_nodes += [r["dec"].node_features(r["ws_d"], b, l) for l in range(r["dec"].n_levels + 1)]
    for i, (mine, ref) in enumerate(zip(mine_nodes, g["nodes_all"])):
        for key, val in ref.items():
            errs[f"nodes_all[{i}]{key}"] = rel_err(mine[eval(key)], val)
    errs["latent00"] = rel_err(r["lat00"], g["latent"]["(0, 0)"])
    errs["latent11"] = rel_err(r["lat11"], g["latent"]["(1, 1)"])
    errs["recons"] = rel_err(r["recon"], g["recons"])
    errs["gen00"] = rel_err(r["gen00"], g["generated"]["(0, 0)"])
    print(name, {k: f"{v:.2e}" for k, v in errs.items()})
    bad = {k: v for k, v in errs.items() if not v < 1e-10}
    assert not bad, bad


@pytest.mark.parametrize("name", CASES)
def test_loss_and_gradients_match_reference(name):
    from lgn_autoencoder_b200 import fused
    dev = torch.device("cuda:0")
    g = load_golden(name)
    r = _run(g, dev)
    recon = r["recon"].clone().requires_grad_(True)
    loss = fused.chamfer_loss(recon, r["p4"], "sum")
    l1 = 1e-8 * (r["th_e"].abs().sum() + r["th_d"].abs().sum())
    assert abs((loss + l1).item() - g["loss"].item()) < 1e-11 * abs(g["loss"].item())
    loss.backward()
    g_lat11, gth_d = fused.decoder_backward_raw(r["dec"], r["th_d"], r["lat11"], r["ws_d"], recon.grad.contiguous(), None)
    gth_e = fused.encoder_backward_raw(r["enc"], r["th_e"], r["p4"], r["mask"], r["ws_e"], r["sel"], None, g_lat11)
    torch.cuda.synchronize()
    mine_e = {k: v + 1e-8 * torch.sign(g["enc_state"][k].to(dev)) for k, v in r["enc"].views(gth_e).items()}
    mine_d = {k: v + 1e-8 * torch.sign(g["dec_state"][k].to(dev)) for k, v in r["dec"].views(gth_d).items()}
    for nm, mine, ref in (("enc", mine_e, g["grads_enc"]), ("dec", mine_d, g["grads_dec"])):
        errs = grad_errors(mine, ref)
        worst = sorted(errs.items(), key=lambda kv: -kv[1][0])[:5]
        print(name, nm, [(k, f"{e[0]:.1e}", f"{e[1]:.1e}") for k, e in worst])
    assert_grads_close(mine_d, g["grads_dec"])
    assert_grads_close(mine_e, g["grads_enc"])
