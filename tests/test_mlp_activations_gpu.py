"""Every CGMLP activation of the reference's table (leakyrelu, relu, elu, sigmoid, logsigmoid, tanh, atan) on the fused path.

The oracle's CGMLP applies LeakyReLU(0.01); these tests run it with the activation under test (the `oracle_activation` fixture
replaces its `cgmlp`), and run the modules with the layer-level composite disabled (`fused_only`), so whatever runs, runs on the
fused kernels.  Acceptance as in tests/test_fused_coverage_gpu.py: latent, reconstruction and loss within 1e-10 relative of the
oracle; every parameter gradient within 1e-10 * max(|ref|, 1e-4 * gmax).  LeakyReLU is the control."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests.helpers import rel_err
from tests.test_fused_coverage_gpu import _assert_forward, _assert_grads, _jets, _oracle_step
from tests.test_input_grad_gpu import _module_run, _oracle_p4_grad, zero_mass_rule  # noqa: F401  (fixture)

# The reference's activations (lgn/nn/generic_levels.py:119-135) with torch's default parameters.
ORACLE_ACTS = {
    "leakyrelu": lambda x: F.leaky_relu(x, 0.01),
    "relu": torch.relu,
    "elu": F.elu,
    "sigmoid": torch.sigmoid,
    "logsigmoid": F.logsigmoid,
    "tanh": torch.tanh,
    "atan": torch.atan,
}
ACTS = list(ORACLE_ACTS)
CODES = {"leakyrelu": 0, "relu": 1, "elu": 2, "sigmoid": 3, "logsigmoid": 4, "tanh": 5, "atan": 6}   # LGAE_ACT_*
UNSUPPORTED = -2   # LGAE_E_UNSUPPORTED

CASES = {
    # per-lane adjoint; 60 rows (not a multiple of 8); hidden widths 24 and 18 (not a multiple of 8); two hidden layers
    "n30": dict(seed=51, batch=2, n=30, num_basis_fn=3, enc_channels=[3, 4, 3], dec_channels=[4, 3, 4], tau_s=1, tau_v=2,
                map_to_latent="mean", mlp_depth=2, mlp_width=3, pad=True),
    # tiled adjoint at N = 40 with padded jets; hidden widths 8 and 12 / 16
    "n40_tiled": dict(seed=52, batch=3, n=40, num_basis_fn=4, enc_channels=[2, 4, 2], dec_channels=[3, 2, 4], tau_s=1, tau_v=2,
                      map_to_latent="min&max", mlp_depth=2, mlp_width=2, pad=True),
    # NTI = 1 at the widest hidden layers the fused MLP takes: 36 (C' = 3) and 48 (C' = 4); 39 rows
    "w36_w48": dict(seed=53, batch=3, n=13, num_basis_fn=5, enc_channels=[2, 3, 4], dec_channels=[4, 4, 3], tau_s=1, tau_v=2,
                    map_to_latent="sum", mlp_depth=1, mlp_width=6, pad=True),
    # NTI = 2: 5-8 output channels (2C' = 10..16 inputs, hidden widths 20-32); 22 rows
    "nti2": dict(seed=54, batch=2, n=11, num_basis_fn=3, enc_channels=[5, 6, 8], dec_channels=[6, 7, 5], tau_s=1, tau_v=2,
                 map_to_latent="max", mlp_depth=2, mlp_width=2, pad=False),
}


@pytest.fixture
def fused_only(monkeypatch):
    """The modules' layer-level composite raises."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder

    def composite(*args, **kwargs):
        raise AssertionError("the layer-level composite ran")

    monkeypatch.setattr(LGNEncoder, "_forward_generic", composite)
    monkeypatch.setattr(LGNDecoder, "_forward_generic", composite)


@pytest.fixture
def oracle_activation(monkeypatch):
    """Call with an activation name: the oracle's CGMLP uses that activation from then on."""
    from oracle import lgae_oracle as orc

    def use(name):
        act = ORACLE_ACTS[name]

        def cgmlp(rep, linears, negative_slope=0.01):
            x = rep.pop((0, 0)).squeeze(-1)
            s = x.shape
            x = x.permute(1, 2, 3, 0).contiguous().view(s[1:3] + (2 * s[3],))
            for w, b in linears[:-1]:
                x = act(F.linear(x, w, b))
            w, b = linears[-1]
            x = F.linear(x, w, b)
            rep[(0, 0)] = x.view(s[1:] + (2,)).permute(3, 0, 1, 2).unsqueeze(-1)
            return rep

        monkeypatch.setattr(orc, "cgmlp", cgmlp)

    return use


def _build(cfg, dev, activation, mlp_depth=None):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg["seed"])
    depth = cfg["mlp_depth"] if mlp_depth is None else mlp_depth
    common = dict(maxdim=[2], num_basis_fn=cfg["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation=activation,
                  mlp=True, mlp_depth=depth, mlp_width=cfg["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=cfg["tau_s"],
                     tau_latent_vectors=cfg["tau_v"], num_channels=cfg["enc_channels"], jet_features=False,
                     map_to_latent=cfg["map_to_latent"], **common)
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=cfg["tau_s"] * mult, tau_latent_vectors=cfg["tau_v"] * mult, num_output_particles=cfg["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=cfg["dec_channels"], cg_dict=enc.cg_dict, **common)
    return enc.to(dev), dec.to(dev)


def _grads(models):
    return {kind: {k: p.grad.detach().clone() for k, p in m.named_parameters()} for kind, m in models.items()}


# ---------------------------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("activation", ACTS)
def test_activation_is_fused_with_its_descriptor_code(activation):
    enc, dec = _build(CASES["n30"], torch.device("cpu"), activation)
    assert enc.fused and dec.fused, (enc._fused_reason, dec._fused_reason)
    assert enc._plan.desc.mlp_activation == CODES[activation] == dec._plan.desc.mlp_activation
    upper, _ = _build(CASES["n30"], torch.device("cpu"), activation.upper())
    assert upper._plan.desc.mlp_activation == CODES[activation]


def test_descriptor_codes_match_the_library_table():
    from lgn_autoencoder_b200 import _lib
    assert _lib.ACTIVATIONS == CODES


@pytest.mark.parametrize("activation", ["leakyrelu", "sigmoid"])
def test_depth_zero_stays_on_the_composite(activation):
    enc, dec = _build(CASES["n30"], torch.device("cpu"), activation, mlp_depth=0)
    assert not enc.fused and not dec.fused
    assert enc._fused_reason == dec._fused_reason == "MLP depth 0"


def test_unknown_activation_raises():
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.nn import get_activation_fn
    with pytest.raises(ValueError):
        get_activation_fn("swish")
    with pytest.raises(ValueError):
        _build(CASES["n30"], torch.device("cpu"), "swish")
    enc, _ = _build(CASES["n30"], torch.device("cpu"), "tanh")
    with pytest.raises(ValueError):
        fused.FusedPlan("encoder", {k: tuple(p.shape) for k, p in enc.named_parameters()}, n_particles=30, channels=[3, 4, 3],
                        num_basis_fn=3, mlp_depth=2, mlp_width=3, activation="swish")


@pytest.mark.parametrize("code", [7, -1])
def test_out_of_range_code_is_refused_before_any_launch(code):
    """A descriptor with an activation code outside LGAE_ACT_*: the size queries return a negative value and the training steps
    and the MLP entry point refuse with LGAE_E_UNSUPPORTED without touching their (fake) pointers."""
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    enc, dec = _build(CASES["n30"], torch.device("cpu"), "leakyrelu")
    ok_e, ok_d = C.byref(enc._plan.desc), C.byref(dec._plan.desc)
    assert lib.lgae_workspace_doubles(ok_e, 4) > 0 and lib.lgae_train_step_partials_doubles(ok_e, ok_d, 4) > 0
    for plan in (enc._plan, dec._plan):
        plan.desc.mlp_activation = code
    de, dd = C.byref(enc._plan.desc), C.byref(dec._plan.desc)
    assert lib.lgae_workspace_doubles(de, 4) == -1 and lib.lgae_partials_doubles(dd, 4) == -1
    assert lib.lgae_mlp_pack_doubles(de, 0) == -1
    assert lib.lgae_train_step_partials_doubles(de, dd, 4) == -1
    assert lib.lgae_train_step_tiled_scratch_doubles(de, dd, 4) < 0
    fake = C.c_void_p(0x1000)
    off_d = enc._plan.n_params + 4
    args = [fake] * 3 + [None, 2, 0] + [fake] * 13 + [off_d, fake, 0.0, 0, 0, None]
    assert lib.lgae_train_step(de, dd, *args) == UNSUPPORTED
    assert lib.lgae_train_step_tiled(de, dd, *args) == UNSUPPORTED
    assert lib.lgae_mlp_forward(de, 0, fake, fake, 8, fake, fake, fake, None) == UNSUPPORTED
    # without an MLP the field is not read
    for plan in (enc._plan, dec._plan):
        plan.desc.has_mlp = 0
    assert lib.lgae_workspace_doubles(de, 4) > 0


@pytest.mark.parametrize("activation", ACTS)
def test_oracle_table_matches_get_activation_fn(activation):
    from lgn_autoencoder_b200.nn import get_activation_fn
    torch.manual_seed(0)
    x = torch.cat([torch.randn(4096, dtype=torch.float64) * 6, torch.tensor([0.0, -0.0, 1e-300, -40.0, 40.0], dtype=torch.float64)])
    assert torch.equal(get_activation_fn(activation)(x), ORACLE_ACTS[activation](x)), activation


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("activation", ACTS)
def test_module_matches_oracle(activation, case, fused_only, oracle_activation):
    """Module forward + autograd backward (per-lane at N <= 32, tiled above) against one oracle step; the gradients are
    bit-identical on a second run."""
    from lgn_autoencoder_b200 import fused
    oracle_activation(activation)
    cfg = CASES[case]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev, activation)
    assert enc.fused and dec.fused
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 1e-8)
    batch = {k: v.to(dev) for k, v in batch_cpu.items() if k in ("p4", "labels")}
    runs = []
    for _ in range(2):
        for m in (enc, dec):
            m.zero_grad(set_to_none=True)
        latent = enc(batch)
        recon = dec(latent)
        loss = fused.chamfer_loss(recon, batch["p4"], "sum") + 1e-8 * (enc.l1_norm() + dec.l1_norm())
        loss.backward()
        runs.append((loss.item(), recon.detach().clone(), _grads(models)))
    lat = {key: latent[key].detach() for key in ((0, 0), (1, 1))}
    what = f"{activation}/{case}"
    _assert_forward(what, lat, recon.detach(), runs[0][0], ref_latent, ref_recon, ref_loss.item())
    _assert_grads(what, models, runs[0][2], ref_grads)
    (la, ra, ga), (lb, rb, gb) = runs
    assert la == lb and torch.equal(ra, rb), what
    for kind in ga:
        for k in ga[kind]:
            assert torch.equal(ga[kind][k], gb[kind][k]), (what, kind, k)


@pytest.mark.gpu
@pytest.mark.parametrize("adjoint", ["per_lane", "tiled"])
@pytest.mark.parametrize("activation", ACTS)
def test_train_step_matches_oracle(activation, adjoint, fused_only, oracle_activation):
    """FusedTrainStep graph-replayed and eager against one oracle step; the two agree bit for bit."""
    from lgn_autoencoder_b200.train import FusedTrainStep
    oracle_activation(activation)
    cfg = CASES["n30" if adjoint == "per_lane" else "n40_tiled"]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev, activation)
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 1e-8)
    p4 = batch_cpu["p4"].to(dev)
    labels = batch_cpu["labels"].to(dev) if cfg["pad"] else None
    results = []
    for use_graph in (True, False):
        step = FusedTrainStep(enc, dec, cfg["batch"], l1_lambda=1e-8, normalize=False, use_labels=cfg["pad"], use_graph=use_graph,
                              get_real="sum", adjoint=adjoint)
        for _ in range(2):   # graph: capture, then a replay
            loss = step.step(p4, labels).item()
        torch.cuda.synchronize()
        what = f"{activation}/{adjoint}/{'graph' if use_graph else 'eager'}"
        lat = {(0, 0): step.latent00, (1, 1): step.latent11}
        _assert_forward(what, lat, step.recon, loss, ref_latent, ref_recon, ref_loss.item())
        _assert_grads(what, models, _grads(models), ref_grads)
        results.append((loss, step.recon.clone(), step.latent11.clone(), step.g_all.clone()))
    (la, ra, za, ga), (lb, rb, zb, gb) = results
    assert la == lb and torch.equal(ra, rb) and torch.equal(za, zb) and torch.equal(ga, gb), (activation, adjoint)


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ACTS)
def test_inference_at_150_particles_matches_module(activation, fused_only):
    from lgn_autoencoder_b200.train import FusedInference
    cfg = dict(CASES["n40_tiled"], n=150, batch=4, seed=55)
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev, activation)
    batch = {k: v.to(dev) for k, v in _jets(cfg, cfg["batch"]).items() if k in ("p4", "labels")}
    with torch.no_grad():
        latent = enc(batch)
        recon = dec(latent)
    inf = FusedInference(enc, dec, cfg["batch"], normalize=False, use_labels=True, get_real="sum")
    for _ in range(2):
        inf.score(batch["p4"], batch["labels"])
    torch.cuda.synchronize()
    assert rel_err(inf.recon, recon) < 1e-10, activation
    assert rel_err(inf.latent11, latent[(1, 1)].reshape(inf.latent11.shape)) < 1e-10, activation


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["n30", "n40_tiled"])
@pytest.mark.parametrize("activation", ["sigmoid", "elu"])
def test_p4_grad_matches_oracle(activation, case, fused_only, oracle_activation, zero_mass_rule):
    oracle_activation(activation)
    cfg = CASES[case]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev, activation)
    batch = {k: v for k, v in _jets(cfg, cfg["batch"]).items() if k in ("p4", "labels")}
    g_p4, grads = _module_run(enc, dec, batch, "sum", True)
    _, grads_ref = _module_run(enc, dec, batch, "sum", False)
    ref = _oracle_p4_grad(enc, dec, cfg, batch, "sum")
    err = rel_err(g_p4, ref)
    assert err <= 1e-10, (activation, case, err)
    for k in grads:
        assert torch.equal(grads[k], grads_ref[k]), (activation, case, k)


def _raw_rows(k):
    return 8 * torch.cuda.get_device_properties(0).multi_processor_count * k + 3


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1, 21, "grid"])
@pytest.mark.parametrize("activation", ACTS)
def test_raw_mlp_matches_autograd(activation, rows):
    """lgae_mlp_forward / lgae_mlp_backward on one level (hidden width 18, 6 inputs; two hidden layers) against torch fp64
    autograd, at 1 and 21 rows and at 8 * SMs * 2 + 3 rows (several slabs per CTA, a partial last group)."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200._lib import ptr
    lib = _lib.load()
    dev = torch.device("cuda:0")
    rows = _raw_rows(2) if rows == "grid" else rows
    enc, _ = _build(CASES["n30"], dev, activation)
    desc, level = enc._plan.desc, 1                        # level 1: C' = 3, width 3 * 6 = 18
    theta, _ = enc._flat_params()
    lin = [(m.weight, m.bias) for m in enc.lgn_cg.mlp_levels[level].linear]
    nin, width = lin[0][0].shape[1], lin[0][0].shape[0]
    assert (nin, width) == (6, 18)
    torch.manual_seed(rows)
    x = torch.randn(rows, nin, dtype=torch.float64, device=dev) * 2
    g_y = torch.randn(rows, nin, dtype=torch.float64, device=dev)
    wpack = torch.empty(lib.lgae_mlp_pack_doubles(C.byref(desc), level), dtype=torch.float64, device=dev)
    acts = torch.empty(len(lin) - 1, rows, 8 * ((width + 7) // 8), dtype=torch.float64, device=dev)
    y = torch.empty(rows, nin, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    assert lib.lgae_mlp_forward(C.byref(desc), level, ptr(theta), ptr(x), rows, ptr(wpack), ptr(acts), ptr(y), st) == 0
    g_x = torch.empty_like(x)
    gtheta = torch.zeros_like(theta)
    partials = torch.empty(lib.lgae_partials_doubles(C.byref(desc), 1), dtype=torch.float64, device=dev)
    assert lib.lgae_mlp_backward(C.byref(desc), level, ptr(theta), ptr(x), rows, ptr(wpack), ptr(acts), ptr(g_y), ptr(g_x), ptr(gtheta),
                                 ptr(partials), st) == 0
    torch.cuda.synchronize()

    xr = x.detach().clone().requires_grad_(True)
    params = [(w.detach().clone().requires_grad_(True), b.detach().clone().requires_grad_(True)) for w, b in lin]
    h = xr
    for w, b in params[:-1]:
        h = ORACLE_ACTS[activation](F.linear(h, w, b))
    yr = F.linear(h, *params[-1])
    yr.backward(g_y)
    assert rel_err(y, yr.detach()) < 1e-10, activation
    assert rel_err(g_x, xr.grad) < 1e-10, activation
    names = [n for n, _ in enc.named_parameters() if n.startswith(f"lgn_cg.mlp_levels.{level}.linear.")]
    views = enc._plan.views(gtheta)
    ref = {f"lgn_cg.mlp_levels.{level}.linear.{i}.{'weight' if j == 0 else 'bias'}": t.grad
           for i, pair in enumerate(params) for j, t in enumerate(pair)}
    assert sorted(names) == sorted(ref)
    gmax = max(g.abs().max().item() for g in ref.values())
    for n in names:
        err = (views[n] - ref[n]).abs().max().item()
        assert err <= 1e-10 * max(ref[n].abs().max().item(), 1e-4 * gmax), (activation, n, err)
    # the rest of theta's gradient is untouched
    mask = torch.ones_like(gtheta, dtype=torch.bool)
    for n in names:
        off, cnt, _ = enc._plan.offsets[n]
        mask[off:off + cnt] = False
    assert not gtheta[mask].any()
