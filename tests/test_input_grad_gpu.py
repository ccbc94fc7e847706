"""Gradients with respect to the jets on the fused maxdim-2 path: p4.grad through the encoder adjoints (per-lane at N <= 32, tiled
above), the chamfer loss's target and normalize_p4.

The reference is the CPU oracle's autograd with one deviation, the zero-mass rule (DESIGN.md section 4e): where normsq4(p) == 0
exactly, the mass scalar sqrt|p^2| contributes nothing (the reference gives 0 * inf = NaN there).  The oracle is run with a hook
that zeroes the incoming gradient of normsq4's output where that output is 0.  Acceptance: p4.grad within 1e-10 per-tensor
max-norm relative of the hooked oracle; parameter gradients bit-identical to the same run without p4.requires_grad."""
import ctypes as C

import pytest
import torch

from tests.helpers import load_golden, rel_err

GET_REAL = ("real", "imag", "sum", "mean", "norm")
BADARG = -1   # LGAE_E_BADARG


# -----------------------------------------------------------------------------------------------------------------------------
# helpers
# -----------------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def zero_mass_rule(monkeypatch):
    """The oracle with the zero-mass rule: normsq4's output passes no gradient where it is exactly 0."""
    from oracle import lgae_oracle as orc
    orig = orc.normsq4

    def hooked(p):
        out = orig(p)
        if out.requires_grad:
            zero = out.detach() == 0
            out.register_hook(lambda g: torch.where(zero, torch.zeros_like(g), g))
        return out

    monkeypatch.setattr(orc, "normsq4", hooked)


@pytest.fixture
def fused_only(monkeypatch):
    """The modules' layer-level composite raises: whatever runs, runs on the fused kernels."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder

    def composite(*args, **kwargs):
        raise AssertionError("the layer-level composite ran")

    monkeypatch.setattr(LGNEncoder, "_forward_generic", composite)
    monkeypatch.setattr(LGNDecoder, "_forward_generic", composite)


def _build(cfg, dev, scale=1.0):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg.get("seed", 0))
    common = dict(maxdim=[2], num_basis_fn=cfg.get("num_basis_fn", 10), max_zf=[1], weight_init="randn", level_gain=[1.0],
                  activation="leakyrelu", mlp=True, mlp_depth=cfg.get("mlp_depth", 6), mlp_width=cfg.get("mlp_width", 6),
                  device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=cfg["tau_s"],
                     tau_latent_vectors=cfg["tau_v"], num_channels=cfg["enc_channels"], jet_features=False,
                     map_to_latent=cfg["map_to_latent"], scale=scale, **common)
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=cfg["tau_s"] * mult, tau_latent_vectors=cfg["tau_v"] * mult, num_output_particles=cfg["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=cfg["dec_channels"], cg_dict=enc.cg_dict, **common)
    return enc.to(dev), dec.to(dev)


def _golden(name, dev):
    g = load_golden(name)
    enc, dec = _build(dict(g["cfg"], seed=0), dev)
    enc.load_state_dict(g["enc_state"])
    dec.load_state_dict(g["dec_state"])
    batch = {k: v for k, v in g["batch"].items() if k in ("p4", "labels")}
    return g["cfg"], enc, dec, batch


def _module_run(enc, dec, batch, get_real, want_p4_grad, encoder_only=False, dev=torch.device("cuda:0")):
    """Encoder -> decoder -> fused chamfer against the jets themselves (or, encoder only, the sum of squared latents).
    Returns (p4.grad or None, {name: param.grad})."""
    from lgn_autoencoder_b200 import fused
    for m in (enc, dec):
        m.zero_grad(set_to_none=True)
    p4 = batch["p4"].to(dev).clone().requires_grad_(want_p4_grad)
    data = {"p4": p4}
    if "labels" in batch:
        data["labels"] = batch["labels"].to(dev)
    latent = enc(data)
    if encoder_only:
        loss = (latent[(0, 0)] ** 2).sum() + (latent[(1, 1)] ** 2).sum()
    else:
        loss = fused.chamfer_loss(dec(latent), p4, get_real)
    loss.backward()
    grads = {f"{kind}.{k}": p.grad.detach().clone() for kind, m in (("enc", enc), ("dec", dec)) for k, p in m.named_parameters()
             if p.grad is not None}
    return (p4.grad.detach().clone() if want_p4_grad else None), grads


def _oracle_p4_grad(enc, dec, cfg, batch, get_real, scale=1.0, encoder_only=False):
    from oracle import lgae_oracle as orc
    enc_sd = {k: v.detach().cpu().clone() for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone() for k, v in dec.state_dict().items()}
    ecfg = dict(num_channels=cfg["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent=cfg["map_to_latent"], scale=scale)
    dcfg = dict(num_channels=cfg["dec_channels"], maxdim=[2], max_zf=[1])
    p4 = batch["p4"].detach().cpu().clone().requires_grad_(True)
    data = {"p4": p4}
    if "labels" in batch:
        data["labels"] = batch["labels"].cpu()
    latent = orc.encoder_forward(enc_sd, ecfg, data)
    if encoder_only:
        loss = (latent[(0, 0)] ** 2).sum() + (latent[(1, 1)] ** 2).sum()
    else:
        dec_in = {k: v.squeeze(2) for k, v in latent.items()} if cfg["map_to_latent"] == "sum" else latent
        loss = orc.chamfer_loss(orc.get_real(orc.decoder_forward(dec_sd, dcfg, dec_in), get_real), p4)
    loss.backward()
    return p4.grad


# -----------------------------------------------------------------------------------------------------------------------------
# oracle parity on the golden fixtures
# -----------------------------------------------------------------------------------------------------------------------------
GOLDEN = ["cfg1_b3", "pad_n8", "mean_n6", "minplusmax_n6", "real_n6", "norm_n6", "n40_b2", "sum_n6"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN)
def test_p4_grad_matches_oracle_on_golden_fixtures(name, zero_mass_rule):
    dev = torch.device("cuda:0")
    cfg, enc, dec, batch = _golden(name, dev)
    get_real = cfg.get("get_real", "sum")
    enc_only = bool(cfg.get("encoder_only", False))
    g_p4, grads = _module_run(enc, dec, batch, get_real, True, enc_only)
    _, grads_ref = _module_run(enc, dec, batch, get_real, False, enc_only)
    ref = _oracle_p4_grad(enc, dec, cfg, batch, get_real, encoder_only=enc_only)
    if not enc.fused:
        # 'min+max' pools in the layer-level composite, which follows the reference at zero momenta too (out of scope here)
        zero_rows = (batch["p4"] == 0).all(-1)
        g_p4, ref = g_p4.cpu()[~zero_rows], ref[~zero_rows]
    assert torch.isfinite(g_p4).all(), name
    err = rel_err(g_p4, ref)
    print(name, f"p4.grad rel err {err:.2e}")
    assert err <= 1e-10, (name, err)
    assert grads.keys() == grads_ref.keys()
    for k in grads:
        assert torch.equal(grads[k], grads_ref[k]), (name, k)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pad_n8", "n40_b2"])
def test_zero_momentum_particles_are_finite(name):
    """Without the zero-mass rule the oracle is NaN exactly on the zero-momentum particles; the library is finite everywhere (its
    agreement with the hooked oracle is the test above)."""
    dev = torch.device("cuda:0")
    cfg, enc, dec, batch = _golden(name, dev)
    ref = _oracle_p4_grad(enc, dec, cfg, batch, cfg.get("get_real", "sum"))
    zero_rows = (batch["p4"] == 0).all(-1)
    assert zero_rows.any()
    assert torch.equal(torch.isnan(ref).any(-1), zero_rows)
    assert torch.equal(torch.isnan(ref).all(-1), zero_rows)
    g_p4, _ = _module_run(enc, dec, batch, cfg.get("get_real", "sum"), True)
    assert torch.isfinite(g_p4).all()


# -----------------------------------------------------------------------------------------------------------------------------
# coverage: the six latent maps, the five get_real modes, per-lane and tiled, input scales 1 and 2.5
# -----------------------------------------------------------------------------------------------------------------------------
COVER = {
    "n12_mix_real": dict(seed=81, batch=2, n=12, num_basis_fn=3, enc_channels=[2, 4, 3], dec_channels=[3, 2], tau_s=1, tau_v=2,
                         map_to_latent="mix", mlp_depth=1, mlp_width=1, pad=True, get_real="real", scale=1.0),
    "n30_max_imag": dict(seed=82, batch=2, n=30, num_basis_fn=10, enc_channels=[3, 3, 4, 4], dec_channels=[4, 3], tau_s=1, tau_v=3,
                         map_to_latent="max", mlp_depth=2, mlp_width=2, pad=False, get_real="imag", scale=2.5),
    "n20_sum_sum": dict(seed=83, batch=3, n=20, num_basis_fn=5, enc_channels=[1, 5, 3], dec_channels=[2, 3], tau_s=1, tau_v=2,
                        map_to_latent="sum", mlp_depth=1, mlp_width=2, pad=True, get_real="sum", scale=2.5),
    "n33_minmax_mean": dict(seed=84, batch=2, n=33, num_basis_fn=7, enc_channels=[2, 3, 5], dec_channels=[3, 2], tau_s=1, tau_v=2,
                            map_to_latent="min&max", mlp_depth=1, mlp_width=1, pad=True, get_real="mean", scale=1.0),
    "n64_min_norm": dict(seed=85, batch=2, n=64, num_basis_fn=11, enc_channels=[3, 6, 8], dec_channels=[4, 2], tau_s=2, tau_v=2,
                         map_to_latent="min", mlp_depth=1, mlp_width=1, pad=False, get_real="norm", scale=2.5),
    "n150_mean_real": dict(seed=86, batch=2, n=150, num_basis_fn=10, enc_channels=[3, 3, 4, 4], dec_channels=[4, 4, 3], tau_s=1, tau_v=4,
                           map_to_latent="mean", mlp_depth=2, mlp_width=2, pad=True, get_real="real", scale=1.0),
    "n40_max_sum_scaled": dict(seed=87, batch=2, n=40, num_basis_fn=4, enc_channels=[2, 4], dec_channels=[3, 2], tau_s=1, tau_v=2,
                               map_to_latent="max", mlp_depth=1, mlp_width=1, pad=True, get_real="sum", scale=2.5),
}


def test_coverage_table_reaches_every_mode():
    assert {c["map_to_latent"] for c in COVER.values()} == {"mix", "max", "min", "sum", "mean", "min&max"}
    assert {c["get_real"] for c in COVER.values()} == set(GET_REAL)
    assert {c["n"] <= 32 for c in COVER.values()} == {True, False}
    assert {c["scale"] for c in COVER.values()} == {1.0, 2.5}


def _jets(cfg, batch=None, seed=None, mass_scale=0.05):
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(batch or cfg["batch"], cfg["n"], seed=cfg["seed"] + 1 if seed is None else seed, mass_scale=mass_scale,
                              pad=cfg.get("pad", False))
    return {k: v for k, v in data.items() if k in ("p4", "labels")}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(COVER))
def test_p4_grad_matches_oracle_across_configurations(name, zero_mass_rule, fused_only):
    dev = torch.device("cuda:0")
    cfg = COVER[name]
    enc, dec = _build(cfg, dev, cfg["scale"])
    batch = _jets(cfg)
    g_p4, grads = _module_run(enc, dec, batch, cfg["get_real"], True)
    _, grads_ref = _module_run(enc, dec, batch, cfg["get_real"], False)
    ref = _oracle_p4_grad(enc, dec, cfg, batch, cfg["get_real"], scale=cfg["scale"])
    err = rel_err(g_p4, ref)
    print(name, f"p4.grad rel err {err:.2e}")
    assert err <= 1e-10, (name, err)
    for k in grads:
        assert torch.equal(grads[k], grads_ref[k]), (name, k)


# -----------------------------------------------------------------------------------------------------------------------------
# independent checks: finite differences and equivariance
# -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [10, 40])
def test_p4_grad_matches_central_differences(n, fused_only):
    """Massive jets (m ~ 0.1 U), per-lane (N = 10) and tiled (N = 40) adjoint."""
    from lgn_autoencoder_b200 import fused
    dev = torch.device("cuda:0")
    cfg = dict(seed=91, n=n, num_basis_fn=4, enc_channels=[2, 3, 3], dec_channels=[3, 2], tau_s=1, tau_v=2, map_to_latent="mean",
               mlp_depth=1, mlp_width=1, scale=1.0)
    enc, dec = _build(cfg, dev)
    p4 = _jets(cfg, batch=2, mass_scale=0.1)["p4"].to(dev)

    def loss_of(x):
        return fused.chamfer_loss(dec(enc({"p4": x})), x, "real")

    x = p4.clone().requires_grad_(True)
    loss_of(x).backward()
    g = x.grad.detach()
    gen = torch.Generator().manual_seed(5)
    worst = 0.0
    with torch.no_grad():
        for _ in range(12):
            b, i, mu = (int(torch.randint(2, (1,), generator=gen)), int(torch.randint(n, (1,), generator=gen)),
                        int(torch.randint(4, (1,), generator=gen)))
            h = 1e-6 * max(abs(p4[b, i, mu].item()), 1e-3)
            xp, xm = p4.clone(), p4.clone()
            xp[b, i, mu] += h
            xm[b, i, mu] -= h
            fd = (loss_of(xp).item() - loss_of(xm).item()) / (2 * h)
            worst = max(worst, abs(fd - g[b, i, mu].item()) / g.abs().max().item())
    print(n, f"worst fd deviation {worst:.2e}")
    assert worst < 1e-6, worst


def _lorentz(kind, x):
    import math
    L = torch.eye(4, dtype=torch.float64)
    if kind == "boost":
        g = math.cosh(x)
        s = math.sinh(x)
        L[0, 0] = L[3, 3] = g
        L[0, 3] = L[3, 0] = s
    else:
        c, s = math.cos(x), math.sin(x)
        L[1, 1] = L[2, 2] = c
        L[1, 2], L[2, 1] = -s, s
    return L


@pytest.mark.gpu
def test_p4_grad_is_equivariant(zero_mass_rule):
    """For the invariant loss sum |latent (0,0)|^2: grad(L p) = L^{-T} grad(p); deviation no worse than 3x the oracle's own (floor
    1e-12 of the gradient scale), over rotations and boosts."""
    from oracle import lgae_oracle as orc
    dev = torch.device("cuda:0")
    cfg = dict(seed=93, n=12, num_basis_fn=5, enc_channels=[2, 3, 3], dec_channels=[3, 2], tau_s=2, tau_v=2, map_to_latent="mean",
               mlp_depth=1, mlp_width=1, scale=1.0)
    enc, dec = _build(cfg, dev)
    p4 = _jets(cfg, batch=2, mass_scale=0.1)["p4"]
    enc_sd = {k: v.detach().cpu().clone() for k, v in enc.state_dict().items()}
    ecfg = dict(num_channels=cfg["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent="mean")

    def mine(x):
        x = x.to(dev).clone().requires_grad_(True)
        (enc({"p4": x})[(0, 0)] ** 2).sum().backward()
        return x.grad.cpu()

    def oracle(x):
        x = x.clone().requires_grad_(True)
        (orc.encoder_forward(enc_sd, ecfg, {"p4": x})[(0, 0)] ** 2).sum().backward()
        return x.grad

    g0, r0 = mine(p4), oracle(p4)
    for kind, xs in (("boost", (0.1, 0.5, 1.0)), ("rot", (0.3, 1.2, 2.5))):
        for x in xs:
            L = _lorentz(kind, x)
            pl = p4 @ L.T
            # grad(L p) should equal L^{-T} grad(p)  <=>  L^T grad(L p) == grad(p)
            dev_m = ((mine(pl) @ L) - g0).abs().max().item() / g0.abs().max().item()
            dev_r = ((oracle(pl) @ L) - r0).abs().max().item() / r0.abs().max().item()
            print(kind, x, f"mine {dev_m:.2e} oracle {dev_r:.2e}")
            assert dev_m <= max(3 * dev_r, 1e-12), (kind, x, dev_m, dev_r)


# -----------------------------------------------------------------------------------------------------------------------------
# adjoint agreement, determinism, batches past the persistent grid, launch accounting
# -----------------------------------------------------------------------------------------------------------------------------
def _raw_setup(cfg, batch_size, dev, seed=None):
    from lgn_autoencoder_b200 import fused
    enc, _ = _build(cfg, dev, cfg.get("scale", 1.0))
    data = _jets(cfg, batch=batch_size, seed=seed)
    p4 = data["p4"].to(dev).contiguous()
    mask = (data["labels"] != 0).to(torch.uint8).to(dev).contiguous() if "labels" in data else None
    plan, theta = enc._plan, enc._theta_node().detach()
    lat00, lat11, ws, sel = fused.encoder_forward_raw(plan, theta, p4, mask)
    gen = torch.Generator().manual_seed(7)
    g00 = torch.randn(lat00.shape, generator=gen, dtype=torch.float64).to(dev)
    g11 = torch.randn(lat11.shape, generator=gen, dtype=torch.float64).to(dev)
    return plan, theta, p4, mask, ws, sel, g00, g11


RAW_CFG = dict(seed=95, n=27, num_basis_fn=6, enc_channels=[2, 4, 3], dec_channels=[3, 2], tau_s=1, tau_v=3, map_to_latent="min&max",
               mlp_depth=1, mlp_width=1, pad=True, scale=2.5)


@pytest.mark.gpu
def test_tiled_and_per_lane_adjoints_agree_and_repeat():
    from lgn_autoencoder_b200 import fused
    dev = torch.device("cuda:0")
    plan, theta, p4, mask, ws, sel, g00, g11 = _raw_setup(RAW_CFG, 5, dev)
    gt_l, gp_l = fused.encoder_backward_p4_raw(plan, theta, p4, mask, ws, sel, g00, g11, tiled=False)
    gt_t, gp_t = fused.encoder_backward_p4_raw(plan, theta, p4, mask, ws, sel, g00, g11, tiled=True)
    assert rel_err(gp_t, gp_l) <= 1e-12, rel_err(gp_t, gp_l)
    # parameter gradients: bit-identical to the entry points without the input gradient
    assert torch.equal(gt_l, fused.encoder_backward_raw(plan, theta, p4, mask, ws, sel, g00, g11))
    assert torch.equal(gt_t, fused.encoder_backward_tiled_raw(plan, theta, p4, mask, ws, sel, g00, g11))
    # run to run
    for tiled, ref in ((False, gp_l), (True, gp_t)):
        assert torch.equal(fused.encoder_backward_p4_raw(plan, theta, p4, mask, ws, sel, g00, g11, tiled=tiled)[1], ref)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [27, 45])
def test_batch_past_the_persistent_grid(n):
    """More jets than 4 CTAs per SM: per-jet g_p4 equals that of the same jets in a batch of 8."""
    from lgn_autoencoder_b200 import _lib, fused
    dev = torch.device("cuda:0")
    big = 4 * _lib.load().lgae_device_sm_count() + 37
    cfg = dict(RAW_CFG, n=n)
    plan, theta, p4, mask, ws, sel, g00, g11 = _raw_setup(cfg, big, dev)
    tiled = n > 32
    _, gp_big = fused.encoder_backward_p4_raw(plan, theta, p4, mask, ws, sel, g00, g11, tiled=tiled)
    p8, m8 = p4[:8].contiguous(), (mask[:8].contiguous() if mask is not None else None)
    lat00, lat11, ws8, sel8 = fused.encoder_forward_raw(plan, theta, p8, m8)
    _, gp8 = fused.encoder_backward_p4_raw(plan, theta, p8, m8, ws8, sel8, g00[:, :8].contiguous(), g11[:, :8].contiguous(), tiled=tiled)
    assert (gp_big[:8] - gp8).abs().max().item() <= 1e-14 * gp8.abs().max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("tiled", [False, True])
def test_no_input_gradient_means_the_same_launches(tiled):
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200._lib import ptr
    dev = torch.device("cuda:0")
    lib = _lib.load()
    plan, theta, p4, mask, ws, sel, g00, g11 = _raw_setup(RAW_CFG, 4, dev)
    d = C.byref(plan.desc)
    gtheta = torch.empty(plan.n_params, dtype=torch.float64, device=dev)
    part = plan.tiled_scratch(4, dev) if tiled else plan.partials(4, dev)
    st = torch.cuda.current_stream().cuda_stream
    old = lib.lgae_encoder_backward_tiled if tiled else lib.lgae_encoder_backward
    new = lib.lgae_encoder_backward_tiled_p4 if tiled else lib.lgae_encoder_backward_p4
    args = (d, ptr(theta), ptr(p4), ptr(mask), 4, ptr(ws), ptr(sel), ptr(g00), ptr(g11), ptr(gtheta), ptr(part), 0.0, None)
    n0 = lib.lgae_launch_count()
    assert old(*args, st) == 0
    n1 = lib.lgae_launch_count()
    assert new(*args, None, None, st) == 0
    n2 = lib.lgae_launch_count()
    torch.cuda.synchronize()
    assert n2 - n1 == n1 - n0 > 0


# -----------------------------------------------------------------------------------------------------------------------------
# chamfer target and normalize_p4
# -----------------------------------------------------------------------------------------------------------------------------
def _chamfer_each_direction(x, y):
    """The oracle's chamfer loss with each direction summed on its own: the same value as orc.chamfer_loss where N == M, and
    defined where N != M (orc.chamfer_loss adds the two directions' (B,N) and (B,M) minima element by element)."""
    diffs = -(x.unsqueeze(-2) - y.unsqueeze(-3))
    dist = torch.sum(diffs ** 2, dim=-1)
    return (dist.min(dim=-1).values.sum() + dist.min(dim=-2).values.sum()) / 2


@pytest.mark.gpu
@pytest.mark.parametrize("mode", GET_REAL)
@pytest.mark.parametrize("n,m", [(7, 7), (7, 5), (4, 9)])
def test_chamfer_target_grad_matches_oracle(mode, n, m):
    """dL/dtarget (and dL/drecon) against the oracle's autograd: orc.chamfer_loss where N == M, the same formula with the two
    directions summed separately where N != M; one jet with exact ties in both directions."""
    from lgn_autoencoder_b200 import fused
    from oracle import lgae_oracle as orc
    gen = torch.Generator().manual_seed(11)
    B = 3
    recon = torch.randn(2, B, n, 4, generator=gen, dtype=torch.float64)
    target = torch.randn(B, m, 4, generator=gen, dtype=torch.float64)
    # jet 2: exact ties -- target 0 at the origin, reconstructed particles 0, 1, 3 at the same distance from it (particle 1 equal
    # to particle 0, particle 3 its negative)
    recon[:, 2, 1] = recon[:, 2, 0]
    recon[:, 2, 3] = -recon[:, 2, 0]
    target[2, 0] = 0.0
    r = recon.clone().requires_grad_(True)
    t = target.clone().requires_grad_(True)
    ref_fn = orc.chamfer_loss if n == m else _chamfer_each_direction
    (1.7 * ref_fn(orc.get_real(r, mode), t)).backward()
    dev = torch.device("cuda:0")
    rg, tg = recon.to(dev).requires_grad_(True), target.to(dev).requires_grad_(True)
    (1.7 * fused.chamfer_loss(rg, tg, mode)).backward()
    assert rel_err(tg.grad, t.grad) <= 1e-12, rel_err(tg.grad, t.grad)
    assert rel_err(rg.grad, r.grad) <= 1e-12, rel_err(rg.grad, r.grad)


def test_chamfer_reference_with_separate_directions_is_the_oracle_where_n_equals_m():
    from oracle import lgae_oracle as orc
    gen = torch.Generator().manual_seed(12)
    x = torch.randn(3, 6, 4, generator=gen, dtype=torch.float64)
    y = torch.randn(3, 6, 4, generator=gen, dtype=torch.float64)
    assert abs(_chamfer_each_direction(x, y).item() - orc.chamfer_loss(x, y).item()) <= 1e-13 * orc.chamfer_loss(x, y).item()


@pytest.mark.gpu
def test_normalize_p4_grad_matches_torch_with_ties():
    from lgn_autoencoder_b200 import fused
    from oracle import lgae_oracle as orc
    gen = torch.Generator().manual_seed(13)
    B, N = 3, 9
    p4 = torch.randn(B, N, 4, generator=gen, dtype=torch.float64)
    p4[0, 2, 0], p4[0, 5, 0] = 10.0, -10.0    # two particles share the max |E|
    p4[1, 3, 0], p4[1, 3, 3] = 10.0, -10.0    # |E| = |p_z| inside one particle
    p4[2, 4] = torch.tensor([7.0, -7.0, 7.0, 3.0], dtype=torch.float64)   # both at once: tied components, and ...
    p4[2, 6] = torch.tensor([1.0, 7.0, 0.0, -2.0], dtype=torch.float64)   # ... a second particle at the same max
    w = torch.randn(B, N, 4, generator=gen, dtype=torch.float64)
    v = torch.randn(B, 1, 1, generator=gen, dtype=torch.float64)
    x = p4.clone().requires_grad_(True)
    out, f = orc.normalize_p4_overall_max(x)
    ((out * w).sum() + (f * v).sum()).backward()
    dev = torch.device("cuda:0")
    y = p4.to(dev).requires_grad_(True)
    out_m, f_m = fused.normalize_p4(y)
    ((out_m * w.to(dev)).sum() + (f_m * v.to(dev)).sum()).backward()
    assert rel_err(out_m, out) == 0.0 and rel_err(f_m, f) == 0.0
    assert rel_err(y.grad, x.grad) <= 1e-13, rel_err(y.grad, x.grad)
    # only the factor, only the output
    for use_out, use_f in ((False, True), (True, False)):
        x.grad, y.grad = None, None
        out, f = orc.normalize_p4_overall_max(x)
        out_m, f_m = fused.normalize_p4(y)
        (((out * w).sum() if use_out else 0) + ((f * v).sum() if use_f else 0)).backward()
        (((out_m * w.to(dev)).sum() if use_out else 0) + ((f_m * v.to(dev)).sum() if use_f else 0)).backward()
        assert rel_err(y.grad, x.grad) <= 1e-13, (use_out, use_f, rel_err(y.grad, x.grad))


@pytest.mark.gpu
def test_training_step_normalize_with_raw_p4_grad(zero_mass_rule, fused_only):
    from lgn_autoencoder_b200.train import training_step
    from oracle import lgae_oracle as orc
    dev = torch.device("cuda:0")
    cfg, enc, dec, batch = _golden("pad_n8", dev)
    raw = batch["p4"] * 37.0
    x = raw.to(dev).clone().requires_grad_(True)
    loss, _, _ = training_step(enc, dec, x, labels=batch["labels"].to(dev), l1_lambda=0.0, normalize=True, get_real="real")
    loss.backward()
    enc_sd = {k: v.detach().cpu().clone() for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone() for k, v in dec.state_dict().items()}
    ecfg = dict(num_channels=cfg["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent=cfg["map_to_latent"])
    dcfg = dict(num_channels=cfg["dec_channels"], maxdim=[2], max_zf=[1])
    xr = raw.clone().requires_grad_(True)
    pn, _ = orc.normalize_p4_overall_max(xr)
    ref_loss, _, _ = orc.training_step(enc_sd, dec_sd, ecfg, dcfg, {"p4": pn, "labels": batch["labels"]}, l1_lambda=0.0,
                                       get_real_method="real")
    ref_loss.backward()
    assert torch.isfinite(x.grad).all()
    assert rel_err(x.grad, xr.grad) <= 1e-10, rel_err(x.grad, xr.grad)


# -----------------------------------------------------------------------------------------------------------------------------
# CPU-only: size query and argument checks (nothing is launched)
# -----------------------------------------------------------------------------------------------------------------------------
def _plan(n, **kw):
    from collections import OrderedDict
    from lgn_autoencoder_b200.fused import FusedPlan
    g = load_golden("cfg1_b3")
    cfg = g["cfg"]
    return FusedPlan("encoder", OrderedDict((k, tuple(v.shape)) for k, v in g["enc_state"].items()), n_particles=n,
                     channels=cfg["enc_channels"], latent_mode=cfg["map_to_latent"], tau_s=cfg["tau_s"], tau_v=cfg["tau_v"],
                     num_basis_fn=10, mlp=True, mlp_depth=6, mlp_width=6, **kw)


def test_input_grad_scratch_size_query():
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    p30, p150 = _plan(30), _plan(150)
    n8 = lib.lgae_encoder_input_grad_scratch_doubles(C.byref(p30.desc), 8)
    assert n8 >= 8 * 30 * 4 + 8 * 30 * 4 * 20   # gp, and the per-lane adjoint's gA at Cmax = 4
    assert lib.lgae_encoder_input_grad_scratch_doubles(C.byref(p30.desc), 0) >= 0
    assert lib.lgae_encoder_input_grad_scratch_doubles(C.byref(p150.desc), 8) >= 8 * 150 * 4
    assert lib.lgae_encoder_input_grad_scratch_doubles(C.byref(p30.desc), -1) == -1
    assert lib.lgae_encoder_input_grad_scratch_doubles(None, 8) == -1
    dec_like = _plan(30)
    dec_like.desc.is_decoder = 1
    assert lib.lgae_encoder_input_grad_scratch_doubles(C.byref(dec_like.desc), 8) == -1
    bad = _plan(30)
    bad.desc.channels[1] = 99            # beyond LGAE_MAX_CHANNELS: the adjoint refuses the configuration
    assert lib.lgae_encoder_input_grad_scratch_doubles(C.byref(bad.desc), 8) == -2


def test_new_entry_points_reject_bad_arguments_before_launching():
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    p = _plan(30)
    d = C.byref(p.desc)
    fake = C.c_void_p(16)   # never dereferenced: the argument checks fail first
    for fn in (lib.lgae_encoder_backward_p4, lib.lgae_encoder_backward_tiled_p4):
        # g_p4 without gp_scratch
        assert fn(d, fake, fake, None, 4, fake, fake, fake, fake, fake, fake, 0.0, None, fake, None, None) == BADARG
        # no gtheta
        assert fn(d, fake, fake, None, 4, fake, fake, fake, fake, None, fake, 0.0, None, fake, fake, None) == BADARG
        assert fn(None, fake, fake, None, 4, fake, fake, fake, fake, fake, fake, 0.0, None, fake, fake, None) == BADARG
    assert lib.lgae_chamfer_target_grad(fake, fake, 2, 0, 3, 0, None, fake, None) == BADARG
    assert lib.lgae_chamfer_target_grad(fake, fake, 2, 3, 3, 9, None, fake, None) == BADARG
    assert lib.lgae_chamfer_target_grad(fake, fake, 2, 3, 3, 0, None, None, None) == BADARG
    assert lib.lgae_normalize_p4_backward(fake, 2, 0, None, None, fake, None) == BADARG
    assert lib.lgae_normalize_p4_backward(fake, 2, 3, None, None, None, None) == BADARG
    assert lib.lgae_normalize_p4_backward(None, 2, 3, None, None, fake, None) == BADARG
