"""The tiled fused adjoint (lgae_encoder_backward_tiled / lgae_decoder_backward_tiled): training through the module API with more
than 32 particles per jet, against the CPU oracle (oracle/lgae_oracle.py) and the reference's golden vectors, against the per-lane
adjoint at N <= 32, past the persistent grid, and run to run.

Every GPU test here replaces the layer-level composite (``_forward_generic``) of both modules by a function that raises, so a
passing test proves the fused path ran.  Acceptance, as in tests/test_edge_cases_gpu.py: latent, reconstruction and loss within
1e-10 relative of the oracle; every parameter gradient within 1e-10 * max(|ref|, 1e-4 * gmax)."""
import ctypes as C

import pytest
import torch

from tests.helpers import assert_grads_close, rel_err
from tests.test_fused_coverage_gpu import (GET_REAL, TRAIN_CASES, _assert_forward, _assert_grads, _build, _cfgs, _dispatch_cases, _jets,
                                           _levels, mma_nt, pick_ks)

# Oracle configurations, batch 2-3, N > 32: N = 33 leaves one particle in the last block, 64 fills two, 65 and 150 spill into a
# third and fifth.  Between them: every (NT, KS) of the neighbour kernel and of the radial adjoint, channels 1-8, Cout 5-7, all six
# latent maps, all five get_real modes, padded and unpadded jets, and the cfg-1 model at 150 particles.
TILED_CASES = {
    "n33_ks3_mix": dict(seed=71, batch=2, n=33, num_basis_fn=3, enc_channels=[2, 4, 6, 8, 5], dec_channels=[3, 5, 7, 2], tau_s=1, tau_v=2,
                        map_to_latent="mix", mlp_depth=1, mlp_width=1, pad=True, get_real="real"),
    "n64_ks5_max": dict(seed=72, batch=3, n=64, num_basis_fn=7, enc_channels=[1, 3, 6, 7, 6], dec_channels=[5, 6, 4], tau_s=2, tau_v=2,
                        map_to_latent="max", mlp_depth=1, mlp_width=2, pad=False, get_real="imag"),
    "n65_ks8_minmax": dict(seed=73, batch=2, n=65, num_basis_fn=11, enc_channels=[2, 3, 5, 8, 4], dec_channels=[4, 8, 1], tau_s=1, tau_v=2,
                           map_to_latent="min&max", mlp_depth=1, mlp_width=1, pad=True, get_real="sum"),
    "n40_ks8_min": dict(seed=74, batch=2, n=40, num_basis_fn=16, enc_channels=[8, 4, 6], dec_channels=[7, 2, 3], tau_s=1, tau_v=3,
                        map_to_latent="min", mlp_depth=2, mlp_width=2, pad=False, get_real="mean"),
    "n34_ks3_sum": dict(seed=75, batch=3, n=34, num_basis_fn=1, enc_channels=[3, 5], dec_channels=[6, 5, 2], tau_s=1, tau_v=1,
                        map_to_latent="sum", mlp_depth=1, mlp_width=3, pad=True, get_real="norm"),
    "n65_ks5_mean": dict(seed=76, batch=2, n=65, num_basis_fn=10, enc_channels=[2, 5, 7], dec_channels=[3, 6], tau_s=1, tau_v=2,
                         map_to_latent="mean", mlp_depth=1, mlp_width=1, pad=False, get_real="real"),
    "cfg1_n150": dict(seed=77, batch=2, n=150, num_basis_fn=10, enc_channels=[3, 3, 4, 4], dec_channels=[4, 4, 3, 3], tau_s=1, tau_v=8,
                      map_to_latent="min&max", mlp_depth=6, mlp_width=6, pad=True, get_real="real"),
}

# Past the persistent grid (4 CTAs per SM) of the mix and neighbour kernels, whose units are (jet, block of 32) pairs, and of the
# decoder's closed form (one jet per CTA).
CAP_CASE = dict(seed=78, n=40, num_basis_fn=4, enc_channels=[2, 5, 3], dec_channels=[3, 6, 2], tau_s=1, tau_v=2, map_to_latent="mean",
                mlp_depth=1, mlp_width=1, pad=True)
CAP_EXTRA = 37


@pytest.fixture
def fused_only(monkeypatch):
    """The modules' layer-level composite raises: whatever runs, runs on the fused kernels."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder

    def composite(*args, **kwargs):
        raise AssertionError("the layer-level composite ran")

    monkeypatch.setattr(LGNEncoder, "_forward_generic", composite)
    monkeypatch.setattr(LGNDecoder, "_forward_generic", composite)


def _oracle_step(enc, dec, cfg, batch_cpu, get_real, l1_lambda):
    from oracle import lgae_oracle as orc
    enc_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in dec.state_dict().items()}
    ecfg, dcfg = _cfgs(cfg)
    data = {k: v for k, v in batch_cpu.items() if k in ("p4", "labels")}
    latent = orc.encoder_forward(enc_sd, ecfg, data)
    dec_in = {k: v.squeeze(2) for k, v in latent.items()} if cfg["map_to_latent"] == "sum" else latent
    recon = orc.decoder_forward(dec_sd, dcfg, dec_in)
    loss = orc.chamfer_loss(orc.get_real(recon, get_real), data["p4"]) + l1_lambda * (orc.l1_norm(enc_sd) + orc.l1_norm(dec_sd))
    loss.backward()
    grads = {"enc": {k: v.grad for k, v in enc_sd.items()}, "dec": {k: v.grad for k, v in dec_sd.items()}}
    return loss.detach(), {k: v.detach() for k, v in latent.items()}, recon.detach(), grads


def _module_step(enc, dec, batch, get_real, l1_lambda):
    from lgn_autoencoder_b200 import fused
    for m in (enc, dec):
        m.zero_grad(set_to_none=True)
    latent = enc(batch)
    recon = dec(latent)
    loss = fused.chamfer_loss(recon, batch["p4"], get_real) + l1_lambda * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    grads = {kind: {k: p.grad.detach().clone() for k, p in m.named_parameters()} for kind, m in (("enc", enc), ("dec", dec))}
    return {key: latent[key].detach() for key in ((0, 0), (1, 1))}, recon.detach(), loss.item(), grads


# ---------------------------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_tiled_tables_reach_every_specialisation():
    """The oracle configurations reach every (NT, KS) instance of level_bwd_nbr_tiled and radial_bwd_tiled_kernel (the same
    dispatch rule as the radial forward: nt = (4 C + 7) / 8, KS from K = 2 num_basis_fn), channel counts 1-8, Cout 5-7, the six
    latent maps, the five get_real modes, padded and unpadded jets, blocks ending at 1, 0 and 2 particles and the cfg-1 model at 150
    particles; the library instantiates every such (NT, KS) pair."""
    all_nt_ks = {(nt, ks) for nt in (1, 2, 3, 4) for ks in (3, 5, 8)}
    reached, chans, couts, latent, modes, tails = set(), set(), set(), set(), set(), set()
    for cfg in TILED_CASES.values():
        assert 2 <= cfg["batch"] <= 3 and cfg["n"] > 32
        reached |= {(mma_nt(c), pick_ks(2 * cfg["num_basis_fn"])) for c, _ in _levels(cfg, "enc")}
        for kind in ("enc", "dec"):
            for c, cout in _levels(cfg, kind):
                chans |= {c, cout}
                couts.add(cout)
        latent.add(cfg["map_to_latent"])
        modes.add(cfg["get_real"])
        tails.add(cfg["n"] % 32)
    assert reached == all_nt_ks, all_nt_ks - reached
    assert chans >= set(range(1, 9)) and couts >= {5, 6, 7}
    from lgn_autoencoder_b200._lib import LATENT_MODES
    assert latent == {m for m in LATENT_MODES if m != "average"}
    assert modes == set(GET_REAL)
    assert {cfg["pad"] for cfg in TILED_CASES.values()} == {True, False}
    assert tails >= {0, 1, 2}
    cfg1 = TILED_CASES["cfg1_n150"]
    assert (cfg1["n"], cfg1["enc_channels"], cfg1["dec_channels"], cfg1["map_to_latent"], cfg1["mlp_depth"], cfg1["mlp_width"]) == \
        (150, [3, 3, 4, 4], [4, 4, 3, 3], "min&max", 6, 6)
    assert _dispatch_cases("lgae_level.cu", "LGAE_CASE") >= all_nt_ks
    assert _dispatch_cases("lgae_radial.cu", "LGAE_CASE") >= all_nt_ks


def _enc_plan(n, channels, latent_mode, tau_s, tau_v):
    from lgn_autoencoder_b200.models import LGNEncoder
    enc = LGNEncoder(num_input_particles=n, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=tau_s, tau_latent_vectors=tau_v,
                     num_channels=channels, maxdim=[2], num_basis_fn=10, max_zf=[1], weight_init="randn", level_gain=[1.0],
                     activation="leakyrelu", mlp=True, mlp_depth=1, mlp_width=1, jet_features=False, map_to_latent=latent_mode,
                     device=torch.device("cpu"), dtype=torch.float64)
    return enc


def test_tiled_scratch_query_and_routing_without_gpu():
    """lgae_backward_tiled_scratch_doubles: -1 for bad arguments, -2 for a configuration the tiled adjoint cannot run (the 'mix'
    latent adjoint over 150 x 8 inputs does not fit its shared memory), otherwise a size that grows with the batch; the module
    records the refusal in _tiled_reason and keeps routing that configuration's training to the composite."""
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    enc = _enc_plan(150, [3, 3, 4, 4], "min&max", 1, 8)
    d = C.byref(enc._plan.desc)
    assert enc._tiled_reason is None
    n1, n8 = lib.lgae_backward_tiled_scratch_doubles(d, 1), lib.lgae_backward_tiled_scratch_doubles(d, 8)
    assert 0 < n1 < n8
    # gA (B N C 10 complex) and dL/dR of one level (B * 5 blocks * N * C * 128) are both in
    assert n8 >= 8 * 150 * 4 * 20 + 8 * 5 * 150 * 4 * 128
    assert lib.lgae_backward_tiled_scratch_doubles(d, -1) == -1
    assert lib.lgae_backward_tiled_scratch_doubles(None, 4) == -1
    assert lib.lgae_backward_tiled_scratch_doubles(C.byref(_lib.LgaeModelDesc()), 4) == -1
    mix = _enc_plan(150, [2, 8], "mix", 1, 2)
    assert mix.fused and lib.lgae_backward_tiled_scratch_doubles(C.byref(mix._plan.desc), 4) == -2
    assert mix._tiled_reason is not None
    # the size query does not touch the existing geometry
    assert lib.lgae_partials_doubles(d, 8) > 0 and lib.lgae_workspace_offset(d, 8, 7, 0) == -1


def test_decoder_backward_refuses_more_than_32_particles_before_any_launch():
    """lgae_decoder_backward (per-lane adjoint) with N = 40: LGAE_E_UNSUPPORTED before anything is launched (the fake pointers are
    never dereferenced); the tiled entry points refuse a refused configuration the same way."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.models import LGNDecoder
    lib = _lib.load()
    dec = LGNDecoder(tau_latent_scalars=2, tau_latent_vectors=16, num_output_particles=40, tau_output_scalars=1, tau_output_vectors=1,
                     num_channels=[4, 4, 3, 3], maxdim=[2], num_basis_fn=10, max_zf=[1], weight_init="randn", level_gain=[1.0],
                     activation="leakyrelu", mlp=True, mlp_depth=6, mlp_width=6, device=torch.device("cpu"), dtype=torch.float64)
    fake = C.c_void_p(0x1000)
    assert lib.lgae_decoder_backward(C.byref(dec._plan.desc), fake, fake, 2, fake, fake, None, fake, fake, fake, 0.0, None, None) == -2
    mix = _enc_plan(150, [2, 8], "mix", 1, 2)
    assert lib.lgae_encoder_backward_tiled(C.byref(mix._plan.desc), fake, fake, None, 2, fake, None, None, fake, fake, fake, 0.0, None,
                                           None) == -2


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_reference_golden_n40(fused_only):
    """tests/golden/n40_b2.pt (the unmodified reference at 40 particles): forward, loss and every gradient through the module API."""
    from lgn_autoencoder_b200 import fused
    from tests.test_models_gpu import load
    dev = torch.device("cuda:0")
    g, enc, dec, batch = load("n40_b2", dev)
    assert enc._tiled_reason is None and dec._tiled_reason is None
    latent = enc(batch)
    recon = dec(latent)
    for key, val in g["latent"].items():
        assert rel_err(latent[eval(key)], val) < 1e-10, key
    assert rel_err(recon, g["recons"]) < 1e-10
    loss = fused.chamfer_loss(recon, batch["p4"], g["cfg"].get("get_real", "sum")) + 1e-8 * (enc.l1_norm() + dec.l1_norm())
    assert abs(loss.item() - g["loss"].item()) < 1e-10 * abs(g["loss"].item())
    loss.backward()
    assert_grads_close({k: p.grad for k, p in dec.named_parameters()}, g["grads_dec"])
    assert_grads_close({k: p.grad for k, p in enc.named_parameters()}, g["grads_enc"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TILED_CASES))
def test_tiled_configs_match_oracle(name, fused_only):
    """Module API + autograd with N > 32 against one oracle step (its get_real mode, L1 1e-8)."""
    cfg = TILED_CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    assert enc._tiled_reason is None and dec._tiled_reason is None
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, cfg["get_real"], 1e-8)
    batch = {k: v.to(dev) for k, v in batch_cpu.items() if k in ("p4", "labels")}
    lat, recon, loss, grads = _module_step(enc, dec, batch, cfg["get_real"], 1e-8)
    _assert_forward(name, lat, recon, loss, ref_latent, ref_recon, ref_loss.item())
    _assert_grads(name, {"enc": enc, "dec": dec}, grads, ref_grads)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRAIN_CASES))
def test_tiled_matches_per_lane_adjoint(name):
    """N <= 32: both C entry points on the same forward workspace and incoming gradients agree to 1e-12 (each parameter tensor
    relative to max(|per-lane|, 1e-4 * its largest gradient)), latent and input gradients included."""
    from lgn_autoencoder_b200 import fused
    cfg = TRAIN_CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, cfg["batch"]).items() if k in ("p4", "labels")}
    mask = (batch["labels"] != 0).to(torch.uint8).contiguous() if cfg["pad"] else None
    g = torch.Generator(device="cpu").manual_seed(cfg["seed"])
    pe, pd = enc._plan, dec._plan
    with torch.no_grad():
        theta_e, theta_d = enc._flat_params()[0], dec._flat_params()[0]
        lat00, lat11, ws_e, sel = fused.encoder_forward_raw(pe, theta_e, batch["p4"].contiguous(), mask)
        g00 = torch.randn(lat00.shape, generator=g, dtype=torch.float64).to(dev)
        g11 = torch.randn(lat11.shape, generator=g, dtype=torch.float64).to(dev)
        lat_d = torch.randn((2, cfg["batch"], 1, dec.tau_latent_vectors, 4), generator=g, dtype=torch.float64).to(dev)
        recon, _, ws_d = fused.decoder_forward_raw(pd, theta_d, lat_d)
        g_recon = torch.randn(recon.shape, generator=g, dtype=torch.float64).to(dev)

        def close(a, b, what):
            scale = max(b.abs().max().item(), 1e-300)
            for nm, (off, n, _) in pe.offsets.items() if what == "enc" else pd.offsets.items():
                x, y = a[off:off + n], b[off:off + n]
                assert (x - y).abs().max().item() <= 1e-12 * max(y.abs().max().item(), 1e-4 * scale), (name, what, nm)

        ref = fused.encoder_backward_raw(pe, theta_e, batch["p4"], mask, ws_e, sel, g00, g11)
        got = fused.encoder_backward_tiled_raw(pe, theta_e, batch["p4"], mask, ws_e, sel, g00, g11)
        close(got, ref, "enc")
        gl_ref, ref = fused.decoder_backward_raw(pd, theta_d, lat_d, ws_d, g_recon, None)
        gl_got, got = fused.decoder_backward_tiled_raw(pd, theta_d, lat_d, ws_d, g_recon, None)
        close(got, ref, "dec")
        assert (gl_got - gl_ref).abs().max().item() <= 1e-12 * gl_ref.abs().max().item(), name


@pytest.mark.gpu
def test_tiled_batch_past_the_persistent_grid(fused_only):
    """Batch 4 * SMs + 37 at N = 40 (two blocks per jet): the mix and neighbour kernels walk more (jet, block) units than they have
    CTAs, the closed form more jets.  Module API on the full batch against the same jets in chunks whose unit count stays below
    the cap: reconstruction bit-identical, gradient sums within 1e-11."""
    from lgn_autoencoder_b200 import _lib
    cfg = CAP_CASE
    dev = torch.device("cuda:0")
    sms = int(_lib.load().lgae_device_sm_count())
    B = 4 * sms + CAP_EXTRA
    enc, dec = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, B).items() if k in ("p4", "labels")}
    _, recon, _, grads = _module_step(enc, dec, batch, "sum", 0.0)
    chunk = 2 * sms - 1   # 2 blocks per jet: fewer than 4 * SMs units
    acc = {kind: {k: torch.zeros_like(v) for k, v in part.items()} for kind, part in grads.items()}
    for lo in range(0, B, chunk):
        sub = {k: v[lo:lo + chunk] for k, v in batch.items()}
        _, r, _, gr = _module_step(enc, dec, sub, "sum", 0.0)
        assert torch.equal(r, recon[:, lo:lo + chunk]), lo
        for kind in acc:
            for k in acc[kind]:
                acc[kind][k] += gr[kind][k]
    gmax = max(v.abs().max().item() for part in grads.values() for v in part.values())
    for kind in acc:
        for k, v in acc[kind].items():
            assert (v - grads[kind][k]).abs().max().item() <= 1e-11 * gmax, (kind, k)


@pytest.mark.gpu
def test_tiled_adjoint_is_deterministic():
    """Two tiled backward calls on the same workspace give bit-identical gradients (no atomics, fixed summation orders)."""
    from lgn_autoencoder_b200 import fused
    cfg = TILED_CASES["cfg1_n150"]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, 3).items() if k in ("p4", "labels")}
    mask = (batch["labels"] != 0).to(torch.uint8).contiguous()
    g = torch.Generator(device="cpu").manual_seed(5)
    with torch.no_grad():
        theta_e, theta_d = enc._flat_params()[0], dec._flat_params()[0]
        lat00, lat11, ws_e, sel = fused.encoder_forward_raw(enc._plan, theta_e, batch["p4"].contiguous(), mask)
        g11 = torch.randn(lat11.shape, generator=g, dtype=torch.float64).to(dev)
        a = fused.encoder_backward_tiled_raw(enc._plan, theta_e, batch["p4"], mask, ws_e, sel, None, g11)
        b = fused.encoder_backward_tiled_raw(enc._plan, theta_e, batch["p4"], mask, ws_e, sel, None, g11)
        assert torch.equal(a, b)
        recon, _, ws_d = fused.decoder_forward_raw(dec._plan, theta_d, lat11.contiguous())
        g_recon = torch.randn(recon.shape, generator=g, dtype=torch.float64).to(dev)
        la, a = fused.decoder_backward_tiled_raw(dec._plan, theta_d, lat11.contiguous(), ws_d, g_recon, None)
        lb, b = fused.decoder_backward_tiled_raw(dec._plan, theta_d, lat11.contiguous(), ws_d, g_recon, None)
        assert torch.equal(a, b) and torch.equal(la, lb)
