"""Coverage of the fused maxdim-2 path across the kernel specialisations its host code dispatches to, against the CPU oracle
(oracle/lgae_oracle.py, pinned to the reference by tests/test_oracle_golden.py).

The host code picks a template instance from the model's shape: the radial MMA tiling (NT, KS) from the channel count and
the number of radial basis functions, the level adjoint's block size from the channel count, the MLP tiling (ntw, nti) from
the hidden width and the channel count, a latent-map branch, a get_real branch.  The configurations below are chosen so that
between them every instance a module the eligibility checks accept can reach runs at least once, and
``test_config_tables_reach_every_specialisation`` (no GPU needed) restates the dispatch rules and fails if the tables stop
reaching one of them.  A separate test runs batches past the cap of the persistent jet loops (4 CTAs per SM), where a CTA
handles more than one jet.

Acceptance, as in tests/test_edge_cases_gpu.py: latent, reconstruction and loss within 1e-10 relative of the oracle; every
parameter gradient within 1e-10 * max(|ref|, 1e-4 * gmax)."""
import os
import re

import pytest
import torch

from tests.helpers import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lgn_autoencoder_b200", "csrc")

# ---------------------------------------------------------------------------------------------------------------------
# configuration tables
# ---------------------------------------------------------------------------------------------------------------------
# Training configs (batch 2-3, N <= 32): module API + autograd, then the same jets through FusedTrainStep (CUDA graph).
# The comment of each entry says which specialisations it is there for; the coverage guard checks the union.
TRAIN_CASES = {
    # K = 2 (KS 3, one padded slab); encoder levels at NT 1, 2, 3, 4 (per-level radial launches); level adjoints at C = 2, 4,
    # 6, 8 and Cout 5, 6; MLP width 1 x 2C' (C' = 5: width 10, not a multiple of 8); latent 'mix' over 5 channels
    "k2_mix": dict(seed=31, batch=2, n=7, num_basis_fn=1, enc_channels=[2, 4, 6, 8, 5], dec_channels=[3, 5, 7, 2], tau_s=2, tau_v=3,
                   map_to_latent="mix", mlp_depth=1, mlp_width=1, pad=True),
    # K = 6 (KS 3, padded); every encoder level at NT 4: the merged radial launch; N = 32 at C = 8; MLP width 3 x 2C' = 48
    # at C' = 8 (the limit); Cout 7; latent 'sum' over 8 channels; decoder adjoint at C = 4 and C = 8
    "k6_sum_merged_n32": dict(seed=32, batch=2, n=32, num_basis_fn=3, enc_channels=[8, 7, 8], dec_channels=[4, 8, 6], tau_s=1,
                              tau_v=2, map_to_latent="sum", mlp_depth=1, mlp_width=3, pad=True),
    # K = 12 (KS 3, exact slab); N = 31 at C = 8; MLP width 2 x 2C' (ntw 2, 3, 4 / nti 1, 2); latent 'min' over 6 channels
    "k12_min_n31": dict(seed=33, batch=3, n=31, num_basis_fn=6, enc_channels=[3, 4, 8, 6], dec_channels=[6, 3, 1], tau_s=1, tau_v=2,
                        map_to_latent="min", mlp_depth=1, mlp_width=2, pad=False),
    # K = 14 (KS 5, padded); encoder levels at NT 1, 2, 3, 4; MLP width 3 x 2C'; latent 'max' over 6 channels
    "k14_max": dict(seed=34, batch=3, n=12, num_basis_fn=7, enc_channels=[1, 3, 6, 7, 6], dec_channels=[5, 5, 4, 1], tau_s=2, tau_v=2,
                    map_to_latent="max", mlp_depth=2, mlp_width=3, pad=True),
    # K = 22 (KS 8, padded); encoder levels at NT 1, 2, 3; MLP width 4 x 2C' (48 at C' = 6); latent 'min&max'
    "k22_minmax": dict(seed=35, batch=2, n=9, num_basis_fn=11, enc_channels=[2, 4, 5, 6], dec_channels=[6, 5, 3], tau_s=1, tau_v=2,
                       map_to_latent="min&max", mlp_depth=1, mlp_width=4, pad=True),
    # K = 32 (KS 8, exact); encoder levels at NT 4 and 2; MLP width 6 x 2C' (ntw 5, 6 at nti 1); latent 'mean'
    "k32_mean": dict(seed=36, batch=3, n=10, num_basis_fn=16, enc_channels=[8, 4, 3], dec_channels=[7, 3, 4], tau_s=1, tau_v=3,
                     map_to_latent="mean", mlp_depth=1, mlp_width=6, pad=False),
}

# Forward-only configs with N > 32: the encoder levels evaluate the radial functions inside the level kernel, tile by tile
# (level_fwd<true, NT, KS, false>), one CTA per 32 particles; N = 33 leaves one particle in the last tile, N = 64 fills two.
FORWARD_CASES = {
    "n33_ks3": dict(seed=41, batch=2, n=33, num_basis_fn=3, enc_channels=[1, 3, 5, 7, 2], dec_channels=[2, 3, 2], tau_s=1, tau_v=2,
                    map_to_latent="mean", mlp_depth=1, mlp_width=2, pad=False, get_real="real"),
    "n64_ks8": dict(seed=42, batch=2, n=64, num_basis_fn=16, enc_channels=[2, 4, 6, 8, 3], dec_channels=[3, 2, 2], tau_s=1, tau_v=2,
                    map_to_latent="min&max", mlp_depth=1, mlp_width=1, pad=False, get_real="sum"),
    "n65_ks5": dict(seed=43, batch=2, n=65, num_basis_fn=7, enc_channels=[2, 3, 5, 8, 4], dec_channels=[4, 5, 2], tau_s=2, tau_v=2,
                    map_to_latent="max", mlp_depth=1, mlp_width=1, pad=True, get_real="norm"),
}

# Past the grid cap of the persistent jet loops: batch 4 * SMs + 37 (629 on a 148-SM B200), so that some CTAs of the level
# adjoint and of the glue adjoints take a second jet.
CAP_EXTRA = 37
CAP_CASES = {
    "small_channels": dict(seed=51, n=10, num_basis_fn=10, enc_channels=[2, 3, 2], dec_channels=[3, 2, 3], tau_s=1, tau_v=2,
                           map_to_latent="min&max", mlp_depth=1, mlp_width=2, pad=True),
    "wide_channels": dict(seed=52, n=8, num_basis_fn=4, enc_channels=[5, 6, 5], dec_channels=[6, 5, 6], tau_s=1, tau_v=2,
                          map_to_latent="mean", mlp_depth=1, mlp_width=1, pad=False),
}

GET_REAL = ("real", "imag", "sum", "mean", "norm")


def cap_batch(sm_count):
    return 4 * sm_count + CAP_EXTRA


# ---------------------------------------------------------------------------------------------------------------------
# dispatch rules, restated from the host code
# ---------------------------------------------------------------------------------------------------------------------
def mma_nt(c):
    """N-tiles of 8 columns of the radial MMA: 4 outputs (2 radial functions x complex) per channel.
    lgae_radial.cu dispatch_radial (:393) and lgae_level.cu dispatch_level_fwd (:1004): nt = (4 * C + 7) / 8."""
    return (4 * c + 7) // 8


def pick_ks(k):
    """k-steps of the radial MMA for K = 2 * num_basis_fn columns: lgae_radial.cu:364, lgae_level.cu:956."""
    return 3 if k <= 12 else (5 if k <= 20 else (8 if k <= 32 else None))


def level_bwd_branch(c):
    """Block size of the level adjoint: lgae_level.cu launch_level_bwd (:984-989): C <= 3 and C == 4 at 128 threads with their
    own occupancy hints, C >= 5 at 256 threads."""
    return "c<=3" if c <= 3 else ("c==4" if c == 4 else "c>=5")


def mlp_tiles(c_out, mlp_width):
    """(ntw, nti) of the MLP after a level with c_out output channels: lgae_mlp.cu run_mlp (:609-615), nin = 2 * C', hidden width
    mlp_width * 2 * C' (fused.py FusedPlan: d.mlp_width)."""
    return ((mlp_width * 2 * c_out + 7) // 8, (2 * c_out + 7) // 8)


def mlp_admitted():
    """Every (ntw, nti) the modules' eligibility check admits: at most 8 channels, hidden width at most 48 (ntw <= 6);
    lgn_encoder.py / lgn_decoder.py _why_not_fused."""
    return {mlp_tiles(c, w) for c in range(1, 9) for w in range(1, 25) if mlp_tiles(c, w)[0] <= 6}


def _levels(cfg, kind):
    ch = cfg[kind + "_channels"]
    return [(ch[l], ch[l + 1]) for l in range(len(ch) - 1)]


def _dispatch_cases(source, macro):
    with open(os.path.join(CSRC, source)) as f:
        text = f.read()
    return {(int(a), int(b)) for a, b in re.findall(macro + r"\((\d+),\s*(\d+)\)", text)}


def test_config_tables_reach_every_specialisation():
    """No GPU: the tables above reach every radial (NT, KS) pair, both radial launch forms, every tiled level_fwd pair, the
    three level_bwd branches of encoder and decoder, output channels 5-7, every MLP tiling the eligibility check admits, all
    six latent maps (mix / sum / min / max with at least 5 channels), all five get_real modes, N = 31 and 32 at 8 channels and a
    batch past the persistent grid of a 148-SM B200.  Also: the library instantiates a kernel for every tiling the modules can
    ask for, so no accepted model reaches LGAE_E_UNSUPPORTED at run time."""
    all_nt_ks = {(nt, ks) for nt in (1, 2, 3, 4) for ks in (3, 5, 8)}
    radial, merged, per_level = set(), [], []
    bwd = {"enc": set(), "dec": set()}
    couts, mlp, latent_wide, latent = set(), set(), set(), set()
    n_at_c8 = set()
    for name, cfg in TRAIN_CASES.items():
        assert 2 <= cfg["batch"] <= 3 and cfg["n"] <= 32, name
        ks = pick_ks(2 * cfg["num_basis_fn"])
        enc_nts = {mma_nt(c) for c, _ in _levels(cfg, "enc")}
        radial |= {(nt, ks) for nt in enc_nts}
        (merged if len(enc_nts) == 1 else per_level).append(name)
        for kind in ("enc", "dec"):
            for c, cout in _levels(cfg, kind):
                bwd[kind].add(level_bwd_branch(c))
                couts.add(cout)
                mlp.add(mlp_tiles(cout, cfg["mlp_width"]))
        latent.add(cfg["map_to_latent"])
        if cfg["enc_channels"][-1] >= 5:
            latent_wide.add(cfg["map_to_latent"])
        if 8 in cfg["enc_channels"] + cfg["dec_channels"]:
            n_at_c8.add(cfg["n"])
    # radial basis sizes: padded and exact k-slabs of KS 3, 5 and 8
    assert {cfg["num_basis_fn"] for cfg in TRAIN_CASES.values()} >= {1, 3, 6, 7, 11, 16}
    assert radial == all_nt_ks, all_nt_ks - radial
    assert merged and per_level
    assert bwd["enc"] == bwd["dec"] == {"c<=3", "c==4", "c>=5"}, bwd
    assert couts >= {5, 6, 7}
    assert mlp >= mlp_admitted(), mlp_admitted() - mlp
    assert (3, 8) in {(cfg["mlp_width"], c) for cfg in TRAIN_CASES.values() for _, c in _levels(cfg, "enc")}   # width 48 at C' = 8
    assert (1, 5) in {(cfg["mlp_width"], c) for cfg in TRAIN_CASES.values() for _, c in _levels(cfg, "enc")}   # width 10 at C' = 5
    assert latent_wide >= {"mix", "sum", "min", "max"}
    from lgn_autoencoder_b200._lib import LATENT_MODES
    assert latent == {m for m in LATENT_MODES if m != "average"}, latent
    assert n_at_c8 >= {31, 32}
    assert any(cfg["pad"] for cfg in TRAIN_CASES.values()) and not all(cfg["pad"] for cfg in TRAIN_CASES.values())
    # tiled forward (N > 32): every (NT, KS) instance, a last tile of one particle and an exact multiple of 32
    tiled = {(mma_nt(c), pick_ks(2 * cfg["num_basis_fn"])) for cfg in FORWARD_CASES.values() for c, _ in _levels(cfg, "enc")}
    assert tiled == all_nt_ks, all_nt_ks - tiled
    assert {cfg["n"] % 32 for cfg in FORWARD_CASES.values()} >= {0, 1} and min(cfg["n"] for cfg in FORWARD_CASES.values()) > 32
    # get_real
    from lgn_autoencoder_b200.fused import GET_REAL_MODES
    assert set(GET_REAL) == set(GET_REAL_MODES)
    # past the cap: 4 CTAs per SM (lgae_glue.cu glue_grid :1134, lgae_level.cu level_bwd_grid :995)
    assert cap_batch(148) > 4 * 148
    widest = [max(cfg["enc_channels"] + cfg["dec_channels"]) for cfg in CAP_CASES.values()]
    assert min(widest) <= 3 and max(widest) >= 5
    # the library's instance lists cover what the modules can ask for
    assert _dispatch_cases("lgae_mlp.cu", "LGAE_MLP_CASE") >= mlp_admitted()
    assert _dispatch_cases("lgae_radial.cu", "LGAE_CASE") >= all_nt_ks
    assert _dispatch_cases("lgae_level.cu", "LGAE_CASE") >= all_nt_ks


# ---------------------------------------------------------------------------------------------------------------------
# fixtures
# ---------------------------------------------------------------------------------------------------------------------
def _build(cfg, dev):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg["seed"])
    common = dict(maxdim=[2], num_basis_fn=cfg["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu",
                  mlp=True, mlp_depth=cfg["mlp_depth"], mlp_width=cfg["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=cfg["tau_s"],
                     tau_latent_vectors=cfg["tau_v"], num_channels=cfg["enc_channels"], jet_features=False,
                     map_to_latent=cfg["map_to_latent"], **common)
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=cfg["tau_s"] * mult, tau_latent_vectors=cfg["tau_v"] * mult, num_output_particles=cfg["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=cfg["dec_channels"], cg_dict=enc.cg_dict, **common)
    assert enc.fused and dec.fused, (enc._fused_reason, dec._fused_reason)
    return enc.to(dev), dec.to(dev)


def _jets(cfg, batch):
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(batch, cfg["n"], seed=cfg["seed"] + 1, mass_scale=0.05, pad=cfg["pad"])
    if cfg["pad"]:
        # one jet padded completely: every particle masked (labels 0, p4 0)
        data["p4"][0] = 0.0
        data["labels"][0] = 0.0
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    return dict(data, p4=pn)


def _cfgs(cfg):
    ecfg = dict(num_channels=cfg["enc_channels"], maxdim=[2], max_zf=[1], map_to_latent=cfg["map_to_latent"])
    dcfg = dict(num_channels=cfg["dec_channels"], maxdim=[2], max_zf=[1])
    return ecfg, dcfg


def _oracle_step(enc, dec, cfg, batch_cpu, l1_lambda):
    from oracle import lgae_oracle as orc
    enc_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in dec.state_dict().items()}
    ecfg, dcfg = _cfgs(cfg)
    data = {k: v for k, v in batch_cpu.items() if k in ("p4", "labels")}
    latent = orc.encoder_forward(enc_sd, ecfg, data)
    # the reference's 'sum' keeps a spurious axis (lgn_encoder.py:424) that its decoder cannot take; the fused decoder reads the
    # latent as (2,B,1,tau,4), so the oracle's decoder gets it without that axis
    dec_in = {k: v.squeeze(2) for k, v in latent.items()} if cfg["map_to_latent"] == "sum" else latent
    recon = orc.decoder_forward(dec_sd, dcfg, dec_in)
    loss = orc.chamfer_loss(orc.get_real(recon, "sum"), data["p4"])
    if l1_lambda:
        loss = loss + l1_lambda * (orc.l1_norm(enc_sd) + orc.l1_norm(dec_sd))
    loss.backward()
    grads = {"enc": {k: v.grad for k, v in enc_sd.items()}, "dec": {k: v.grad for k, v in dec_sd.items()}}
    return loss.detach(), {k: v.detach() for k, v in latent.items()}, recon.detach(), grads


def _assert_grads(name, models, mine, ref):
    """Every parameter gradient within 1e-10 * max(|ref|, 1e-4 * gmax) (gmax: the largest oracle gradient of both models)."""
    gmax = max(g.abs().max().item() for part in ref.values() for g in part.values() if g is not None)
    for kind, model in models.items():
        for k, _ in model.named_parameters():
            r = ref[kind][k]
            r = torch.zeros_like(mine[kind][k].cpu()) if r is None else r
            err = (mine[kind][k].detach().cpu() - r).abs().max().item()
            assert err <= 1e-10 * max(r.abs().max().item(), 1e-4 * gmax), (name, kind, k, err)


def _assert_forward(name, latent, recon, loss, ref_latent, ref_recon, ref_loss):
    for key in ((0, 0), (1, 1)):
        assert rel_err(latent[key], ref_latent[key]) < 1e-10, (name, key)
    assert rel_err(recon, ref_recon) < 1e-10, name
    assert abs(loss - ref_loss) <= 1e-10 * abs(ref_loss), (name, loss, ref_loss)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRAIN_CASES))
def test_train_configs_match_oracle(name):
    """Module API + autograd, then FusedTrainStep (CUDA graph) on the same weights and jets, against one oracle step."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = TRAIN_CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 1e-8)
    models = {"enc": enc, "dec": dec}

    batch = {k: v.to(dev) for k, v in batch_cpu.items() if k in ("p4", "labels")}
    latent = enc(batch)
    recon = dec(latent)
    loss = fused.chamfer_loss(recon, batch["p4"], "sum") + 1e-8 * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    lat = {key: latent[key].detach() for key in ((0, 0), (1, 1))}
    _assert_forward(name, lat, recon, loss.item(), ref_latent, ref_recon, ref_loss.item())
    _assert_grads(name, models, {kind: {k: p.grad for k, p in m.named_parameters()} for kind, m in models.items()}, ref_grads)

    step = FusedTrainStep(enc, dec, cfg["batch"], l1_lambda=1e-8, normalize=False, use_labels=cfg["pad"], use_graph=True, get_real="sum")
    for _ in range(2):   # capture, then a replay
        l_step = step.step(batch["p4"], batch.get("labels")).item()
    torch.cuda.synchronize()
    lat_step = {(0, 0): step.latent00, (1, 1): step.latent11}
    if cfg["map_to_latent"] == "sum":   # the module keeps the reference's extra axis of 'sum'
        lat_step = {k: v.unsqueeze(-3) for k, v in lat_step.items()}
    _assert_forward(name + "/step", lat_step, step.recon, l_step, ref_latent, ref_recon, ref_loss.item())
    step_grads = {kind: {k: p.grad for k, p in m.named_parameters()} for kind, m in models.items()}
    _assert_grads(name + "/step", models, step_grads, ref_grads)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FORWARD_CASES))
def test_forward_more_than_32_particles_matches_oracle(name):
    """N > 32 forward only: module forward under no_grad and FusedInference (normalisation, encoder, decoder and per-jet chamfer
    in one CUDA graph) against the oracle's forward."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedInference
    from oracle import lgae_oracle as orc
    cfg = FORWARD_CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    raw = orc.synthetic_jets(cfg["batch"], cfg["n"], seed=cfg["seed"] + 1, mass_scale=0.05, pad=cfg["pad"])
    pn, _ = orc.normalize_p4_overall_max(raw["p4"])
    data = dict(raw, p4=pn)
    ecfg, dcfg = _cfgs(cfg)
    enc_sd = {k: v.detach().cpu() for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu() for k, v in dec.state_dict().items()}
    with torch.no_grad():
        ref_latent = orc.encoder_forward(enc_sd, ecfg, {k: v for k, v in data.items() if k in ("p4", "labels")})
        ref_recon = orc.decoder_forward(dec_sd, dcfg, ref_latent)
    x = orc.get_real(ref_recon, cfg["get_real"])
    ref_jet = torch.stack([orc.chamfer_loss(x[b:b + 1], pn[b:b + 1]) for b in range(cfg["batch"])])

    batch = {k: v.to(dev) for k, v in data.items() if k in ("p4", "labels")}
    with torch.no_grad():
        latent = enc(batch)
        recon = dec(latent)
    for key in ((0, 0), (1, 1)):
        assert rel_err(latent[key], ref_latent[key]) < 1e-10, (name, key)
    assert rel_err(recon, ref_recon) < 1e-10, name
    assert rel_err(fused.chamfer_per_jet(recon, batch["p4"], cfg["get_real"]), ref_jet) < 1e-10, name

    labels = raw["labels"].to(dev) if cfg["pad"] else None
    inf = FusedInference(enc, dec, cfg["batch"], normalize=True, use_labels=cfg["pad"], get_real=cfg["get_real"])
    for _ in range(2):
        scores = inf.score(raw["p4"].to(dev), labels).clone()
    torch.cuda.synchronize()
    assert rel_err(inf.latent00, ref_latent[(0, 0)]) < 1e-10 and rel_err(inf.latent11, ref_latent[(1, 1)]) < 1e-10, name
    assert rel_err(inf.recon, ref_recon) < 1e-10, name
    assert rel_err(scores, ref_jet) < 1e-10, name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CAP_CASES))
def test_batch_past_the_persistent_grid(name):
    """Batch 4 * SMs + 37: the level adjoint (lgae_level.cu level_bwd_kernel, jet loop :644) and the glue adjoints
    (lgae_glue.cu enc_latent_bwd_kernel :379, dec_input_bwd_kernel :540, latent_bridge_bwd_kernel :553) loop over more jets than they have CTAs, so some CTAs take a second jet and
    carry their gradient partials across it.  FusedTrainStep on the full batch against the oracle (gradients included), and
    against the same jets in chunks below the cap: per-jet reconstruction and loss bit-identical, gradient sums within 1e-11."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = CAP_CASES[name]
    dev = torch.device("cuda:0")
    sms = int(_lib.load().lgae_device_sm_count())
    B = cap_batch(sms)
    enc, dec = _build(cfg, dev)
    batch_cpu = _jets(cfg, B)
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 0.0)
    models = {"enc": enc, "dec": dec}
    p4 = batch_cpu["p4"].to(dev)
    labels = batch_cpu["labels"].to(dev) if cfg["pad"] else None

    full = FusedTrainStep(enc, dec, B, l1_lambda=0.0, normalize=False, use_labels=cfg["pad"], use_graph=True, get_real="sum")
    for _ in range(2):
        loss = full.step(p4, labels).item()
    torch.cuda.synchronize()
    _assert_forward(name, {(0, 0): full.latent00, (1, 1): full.latent11}, full.recon, loss, ref_latent, ref_recon, ref_loss.item())
    _assert_grads(name, models, {kind: {k: p.grad for k, p in m.named_parameters()} for kind, m in models.items()}, ref_grads)
    g_full, recon, jet_loss = full.g_all.clone(), full.recon.clone(), full.jet_loss.clone()
    assert abs(jet_loss.sum().item() - loss) <= 1e-12 * abs(loss)

    # the same jets in chunks below the cap (every CTA takes at most one jet)
    half = (B + 1) // 2
    assert half < 4 * sms
    g_sum = torch.zeros_like(g_full)
    for lo, hi in ((0, half), (half, B)):
        part = FusedTrainStep(enc, dec, hi - lo, l1_lambda=0.0, normalize=False, use_labels=cfg["pad"], use_graph=False, get_real="sum")
        part.step(p4[lo:hi], None if labels is None else labels[lo:hi])
        torch.cuda.synchronize()
        assert torch.equal(part.recon, recon[:, lo:hi]), (name, lo)
        assert torch.equal(part.jet_loss, jet_loss[lo:hi]), (name, lo)
        g_sum += part.g_all
    assert (g_sum - g_full).abs().max().item() <= 1e-11 * g_full.abs().max().item(), name


@pytest.mark.gpu
@pytest.mark.parametrize("mode", GET_REAL)
def test_get_real_modes_chamfer_and_anomaly_scores(mode):
    """Every get_real mode through the chamfer loss (value and gradient wrt the complex reconstruction) and through the anomaly
    scores, with and without the per-jet rescaling, against orc.get_real + orc.chamfer_loss / orc.anomaly_scores_cartesian
    under fp64 autograd."""
    from lgn_autoencoder_b200 import fused
    from oracle import lgae_oracle as orc
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(61 + GET_REAL.index(mode))
    B, N = 3, 9
    recon_cpu = (torch.rand((2, B, N, 4), generator=g, dtype=torch.float64) - 0.3).requires_grad_(True)
    target = torch.rand((B, N, 4), generator=g, dtype=torch.float64) - 0.3
    factor = torch.rand(B, generator=g, dtype=torch.float64) * 5 + 0.5

    ref = orc.chamfer_loss(orc.get_real(recon_cpu, mode), target)
    ref.backward()
    recon = recon_cpu.detach().to(dev).requires_grad_(True)
    loss = fused.chamfer_loss(recon, target.to(dev), mode)
    loss.backward()
    assert abs(loss.item() - ref.item()) <= 1e-10 * abs(ref.item()), mode
    assert rel_err(recon.grad, recon_cpu.grad) < 1e-10, mode

    x = orc.get_real(recon_cpu.detach(), mode)
    for f in (None, factor):
        fv = 1.0 if f is None else f.view(-1, 1, 1)
        want = orc.anomaly_scores_cartesian(x * fv, target * fv)
        got = fused.anomaly_scores(recon.detach(), target.to(dev), mode, None if f is None else f.to(dev))
        for name in fused.SCORE_NAMES:
            # the Minkowski scores are differences of squares: their error is measured on the Euclidean counterpart's scale
            scale = want[name.replace("lorentz", "cartesian")].abs().max().item()
            assert (got[name].cpu() - want[name]).abs().max().item() <= 1e-10 * scale, (mode, f is not None, name)
