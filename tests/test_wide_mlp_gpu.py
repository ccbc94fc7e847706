"""Scalar MLPs with hidden widths up to 96 on the fused path: the streamed-weight CGMLP kernels (lgae_mlp_streamed.cuh).

The resident MLP kernels keep all layers' weights in shared memory and take hidden widths up to 48 (ntw <= 6, plus (8, 2) and
(9, 2) while the layers fit).  run_mlp (lgae_mlp.cu) runs the streamed kernels exactly where the resident ones have no instance
or need more than 227 KB; a level may therefore run the resident forward and the streamed adjoint.  Acceptance as in
tests/test_fused_coverage_gpu.py: latent, reconstruction and loss within 1e-10 relative of the oracle; every parameter gradient
within 1e-10 * max(|ref|, 1e-4 * gmax); the modules run with the layer-level composite disabled (`fused_only`)."""
import ctypes as C
import os
import re
import types

import pytest
import torch
import torch.nn.functional as F

from tests.helpers import rel_err
from tests.test_fused_coverage_gpu import CSRC, TRAIN_CASES, _assert_forward, _assert_grads, _dispatch_cases, _jets, _oracle_step, mlp_tiles
from tests.test_input_grad_gpu import _module_run, _oracle_p4_grad, zero_mass_rule  # noqa: F401  (fixture)
from tests.test_mlp_activations_gpu import ACTS, ORACLE_ACTS, UNSUPPORTED, fused_only, oracle_activation  # noqa: F401  (fixtures)

SMEM_CAP = 227 * 1024
MLP_BWD_ROWS = 128   # lgae_mlp.cuh

CASES = {
    # the project's wide channel shape: encoder widths 72, 96, 96 / decoder 96, 72, 72 (nti 2); depth 3: the (9, 2) levels run the
    # resident forward and the streamed adjoint, the (12, 2) levels both streamed; padded jets
    "cfg4_shape": dict(seed=71, batch=2, n=12, num_basis_fn=4, enc_channels=[6, 6, 8, 8], dec_channels=[8, 8, 6, 6], tau_s=1, tau_v=2,
                       map_to_latent="min&max", mlp_depth=3, mlp_width=6, pad=True),
    # C' = 5 at mlp_width 5: width 50 (ntw 7, not a multiple of 8), depth 2
    "c5_w50": dict(seed=72, batch=3, n=9, num_basis_fn=3, enc_channels=[3, 5, 5], dec_channels=[5, 5, 2], tau_s=1, tau_v=2,
                   map_to_latent="mean", mlp_depth=2, mlp_width=5, pad=False),
    # C' <= 4 at mlp_width 12: widths 96 (ntw 12) and 72 / 48 at nti 1; 31 particles
    "nti1_w96": dict(seed=73, batch=2, n=31, num_basis_fn=5, enc_channels=[2, 4, 3], dec_channels=[4, 3, 4], tau_s=1, tau_v=2,
                     map_to_latent="max", mlp_depth=2, mlp_width=12, pad=True),
}


# ---------------------------------------------------------------------------------------------------------------------
# the selection rule, restated from lgae_mlp.cu / lgae_mlp.cuh
# ---------------------------------------------------------------------------------------------------------------------
def _frag(layer, n_lin, ntw, nti):
    return (nti if layer == 0 else ntw) * 2 * (nti if layer == n_lin - 1 else ntw) * 32


def mlp_family(ntw, nti, n_lin, bwd):
    """'resident' where lgae_mlp.cu has an LGAE_MLP_CASE instance whose shared memory holds all layers (launch_mlp), else
    'streamed' (7 <= ntw <= 12), else None."""
    wtotal = sum(_frag(layer, n_lin, ntw, nti) for layer in range(n_lin))
    nbytes = 8 * (wtotal + 2 * MLP_BWD_ROWS * (8 * ntw + 4) + 2 * 4 * 8 * ntw if bwd else wtotal + n_lin * 8 * ntw)
    if (ntw, nti) in _dispatch_cases("lgae_mlp.cu", "LGAE_MLP_CASE") and nbytes <= SMEM_CAP:
        return "resident"
    return "streamed" if 7 <= ntw <= 12 and nti in (1, 2) else None


def _kernel_names(ntw, nti, n_lin):
    fwd, bwd = mlp_family(ntw, nti, n_lin, False), mlp_family(ntw, nti, n_lin, True)
    return ("mlp_fwd" if fwd == "resident" else "mlp_fwd_streamed"), ("mlp_bwd" if bwd == "resident" else "mlp_bwd_streamed")


# ---------------------------------------------------------------------------------------------------------------------
# builders
# ---------------------------------------------------------------------------------------------------------------------
def _build(cfg, dev, activation="leakyrelu"):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg["seed"])
    common = dict(maxdim=[2], num_basis_fn=cfg["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation=activation,
                  mlp=True, mlp_depth=cfg["mlp_depth"], mlp_width=cfg["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=cfg["tau_s"],
                     tau_latent_vectors=cfg["tau_v"], num_channels=cfg["enc_channels"], jet_features=False,
                     map_to_latent=cfg["map_to_latent"], **common)
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=cfg["tau_s"] * mult, tau_latent_vectors=cfg["tau_v"] * mult, num_output_particles=cfg["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=cfg["dec_channels"], cg_dict=enc.cg_dict, **common)
    assert enc.fused and dec.fused, (enc._fused_reason, dec._fused_reason)
    return enc.to(dev), dec.to(dev)


# (ntw, nti) -> (C', mlp_width) of a one-level encoder whose MLP has that tiling; widths 54 60 68 78 84 96 / 50 60 72 80 84 90
TILINGS = {(7, 1): (3, 9), (8, 1): (3, 10), (9, 1): (2, 17), (10, 1): (3, 13), (11, 1): (3, 14), (12, 1): (4, 12),
           (7, 2): (5, 5), (8, 2): (5, 6), (9, 2): (6, 6), (10, 2): (5, 8), (11, 2): (7, 6), (12, 2): (5, 9)}


def _one_level(ntw, nti, depth, dev, activation="leakyrelu"):
    c_out, mlp_width = TILINGS[(ntw, nti)]
    assert mlp_tiles(c_out, mlp_width) == (ntw, nti)
    cfg = dict(seed=100 * ntw + nti, n=4, num_basis_fn=2, enc_channels=[2, c_out], dec_channels=[2, 2], tau_s=1, tau_v=1,
               map_to_latent="mean", mlp_depth=depth, mlp_width=mlp_width)
    enc, _ = _build(cfg, dev, activation)
    return enc


def _grads(models):
    return {kind: {k: p.grad.detach().clone() for k, p in m.named_parameters()} for kind, m in models.items()}


# ---------------------------------------------------------------------------------------------------------------------
# no GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_eligibility_is_hidden_width_96():
    """Over C' = 1..8 and mlp_width = 1..24: both models are fused exactly when every level's ntw <= 12."""
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    for c in range(1, 9):
        for w in range(1, 25):
            ok = mlp_tiles(c, w)[0] <= 12
            enc = types.SimpleNamespace(level_maxdim=[2], max_zf=[1], jet_features=False, tau_input_scalars=1, tau_input_vectors=1,
                                        map_to_latent="mean", num_channels=[2, c, 1], mlp=True, mlp_depth=2, mlp_width=w, num_basis_fn=3)
            dec = types.SimpleNamespace(level_maxdim=[2], max_zf=[1], tau_output_scalars=1, tau_output_vectors=1, num_channels=[1, c, 2],
                                        mlp=True, mlp_depth=2, mlp_width=w)
            for reason in (LGNEncoder._why_not_fused(enc), LGNDecoder._why_not_fused(dec)):
                assert reason == (None if ok else "MLP hidden width above 96"), (c, w, reason)
    # a real module at hidden width 104 (C' = 4, mlp_width 13)
    cfg = dict(CASES["nti1_w96"], enc_channels=[2, 4], dec_channels=[4, 2], mlp_width=13)
    with pytest.raises(AssertionError):
        _build(cfg, torch.device("cpu"))


def test_streamed_instances_cover_every_admitted_wide_tiling():
    """The streamed instance list (lgae_mlp_streamed.cuh) and run_mlp's streamed cases (lgae_mlp.cu) cover every tiling with
    ntw >= 7 the modules admit; with the resident instances every admitted tiling has a kernel."""
    admitted = {mlp_tiles(c, w) for c in range(1, 9) for w in range(1, 25) if mlp_tiles(c, w)[0] <= 12}
    wide = {t for t in admitted if t[0] >= 7}
    with open(os.path.join(CSRC, "lgae_mlp_streamed.cuh")) as f:
        text = f.read()
    instances = {(int(a), int(b)) for a, b in re.findall(r"LGAE_MLP_STREAMED_INSTANCE\(EXT,\s*(\d+),\s*(\d+)", text)}
    assert instances >= wide, wide - instances
    with open(os.path.join(CSRC, "lgae_mlp.cu")) as f:
        cases = {int(w) for w in re.findall(r"LGAE_MLP_STREAMED_CASE\((\d+)\)", f.read())}
    assert cases >= {t[0] for t in wide}
    assert admitted <= _dispatch_cases("lgae_mlp.cu", "LGAE_MLP_CASE") | instances
    assert set(TILINGS) == {(w, i) for w in range(7, 13) for i in (1, 2)}


def test_width_104_is_refused_before_any_launch():
    """A descriptor with a hidden width of 104 (ntw 13): every entry point that takes a model descriptor returns
    LGAE_E_UNSUPPORTED without touching its (fake) pointers, and the size queries refuse it."""
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    enc, dec = _build(CASES["nti1_w96"], torch.device("cpu"))
    good_e, good_d = enc._plan.desc, dec._plan.desc
    assert lib.lgae_workspace_doubles(C.byref(good_e), 4) > 0 and lib.lgae_train_step_partials_doubles(C.byref(good_e), C.byref(good_d), 4) > 0
    bad_e, bad_d = type(good_e).from_buffer_copy(good_e), type(good_d).from_buffer_copy(good_d)
    assert bad_e.mlp_width[0] == 96 and bad_d.mlp_width[0] == 72
    bad_e.mlp_width[0] = 104
    bad_d.mlp_width[0] = 104
    fake = C.c_void_p(0x1000)
    checked = 0
    for name, (res, argtypes) in _lib._PROTOS.items():
        n_desc = sum(1 for t in argtypes if t is _lib._D)
        if n_desc == 0:
            continue
        pairs = [(bad_e, good_d), (good_e, bad_d)] if n_desc == 2 else [(bad_e,), (bad_d,)]
        for descs in pairs:
            it = iter(descs)
            args = []
            for t in argtypes:
                if t is _lib._D:
                    args.append(C.byref(next(it)))
                elif t is C.c_int32:
                    args.append(1)
                elif t is C.c_int64:
                    args.append(enc._plan.n_params + 4)
                elif t is C.c_double:
                    args.append(0.0)
                else:
                    args.append(fake)
            if argtypes[-1] is _lib._P:
                args[-1] = None   # the stream
            rc = getattr(lib, name)(*args)
            if res is C.c_int64:
                assert rc < 0, (name, rc)
            else:
                assert rc == UNSUPPORTED, (name, rc)
            checked += 1
    assert checked >= 2 * 20


# lgae_workspace_doubles (enc, dec), lgae_partials_doubles (enc, dec), lgae_backward_tiled_scratch_doubles (enc, dec),
# lgae_train_step_partials_doubles, lgae_train_step_tiled_scratch_doubles at batch 3 and 512, as the parent commit of the streamed
# kernels returned them (148 SMs: the partial rows of the MLP and radial adjoints are one per SM).
PARENT_SIZES = {
    "cfg1": {3: [413744, 171908, 5238044, 3981342, 5140364, 3988542, 9219423, 9121743],
             512: [59340672, 19305216, 5651352, 4865984, 14593512, 6094784, 10523481, 19465641]},
    "k2_mix": {3: [130796, 17212, 307466, 106172, 293258, 109112, 413663, 399455],
               512: [21756672, 2543360, 1707216, 800448, 5911600, 1302208, 2511761, 6716145]},
    "k6_sum_merged_n32": {3: [457872, 75616, 633456, 380888, 679632, 396248, 1014417, 1060593],
                          512: [77101056, 11949568, 1798048, 1280800, 21129216, 3902240, 3091137, 22422305]},
    "k12_min_n31": {3: [438132, 43652, 692604, 29838, 671292, 40998, 722455, 701143],
                    512: [74078720, 7317760, 1647488, 328112, 20308512, 2232752, 1977649, 20638673]},
    "k14_max": {3: [217236, 31780, 1734748, 397756, 1596220, 401356, 2132517, 1993989],
                512: [33491584, 4337920, 2828080, 945440, 9017440, 1559840, 3775569, 9964929]},
    "k22_minmax": {3: [101440, 19240, 929140, 177950, 774036, 181190, 1107127, 952023],
                   512: [16182272, 2717440, 1537904, 696112, 5450728, 1249072, 2240161, 6152985]},
    "k32_mean": {3: [115720, 21208, 988352, 197032, 761024, 201232, 1185433, 958105],
                 512: [19271424, 3141376, 1448488, 587944, 7247720, 1304744, 2044625, 7843857]},
}


def test_size_queries_unchanged():
    from bench import build_models
    from lgn_autoencoder_b200 import _lib
    from tests.test_fused_coverage_gpu import _build as coverage_build
    lib = _lib.load()
    sms = lib.lgae_device_sm_count()
    if sms > 0 and sms != 148:
        pytest.skip(f"sizes recorded for 148 SMs, device has {sms}")
    models = {"cfg1": build_models(torch.device("cpu"))}
    models.update({n: coverage_build(c, torch.device("cpu")) for n, c in TRAIN_CASES.items()})
    assert set(models) == set(PARENT_SIZES)
    for name, (e, d) in models.items():
        de, dd = C.byref(e._plan.desc), C.byref(d._plan.desc)
        for B, want in PARENT_SIZES[name].items():
            got = [lib.lgae_workspace_doubles(de, B), lib.lgae_workspace_doubles(dd, B), lib.lgae_partials_doubles(de, B),
                   lib.lgae_partials_doubles(dd, B), lib.lgae_backward_tiled_scratch_doubles(de, B), lib.lgae_backward_tiled_scratch_doubles(dd, B),
                   lib.lgae_train_step_partials_doubles(de, dd, B), lib.lgae_train_step_tiled_scratch_doubles(de, dd, B)]
            assert got == want, (name, B)


def test_selection_rule_examples():
    """The mixed cases the rule produces: (8, 2) at depth 6 and (9, 2) at depth 5 and 6 fit the resident forward but not its
    adjoint; (9, 2) at depth 7 fits neither; at depth 1 both run resident."""
    assert _kernel_names(8, 2, 7) == ("mlp_fwd", "mlp_bwd_streamed")
    assert _kernel_names(9, 2, 6) == ("mlp_fwd", "mlp_bwd_streamed")
    assert _kernel_names(9, 2, 7) == ("mlp_fwd", "mlp_bwd_streamed")   # 224 KB of forward weights and biases still fit
    assert _kernel_names(9, 2, 8) == ("mlp_fwd_streamed", "mlp_bwd_streamed")
    assert _kernel_names(8, 2, 2) == _kernel_names(9, 2, 2) == ("mlp_fwd", "mlp_bwd")
    assert _kernel_names(12, 2, 7) == ("mlp_fwd_streamed", "mlp_bwd_streamed")
    assert mlp_family(13, 2, 2, False) is None


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the raw MLP entry points
# ---------------------------------------------------------------------------------------------------------------------
def _raw_rows(k):
    return 32 * torch.cuda.get_device_properties(0).multi_processor_count * k + 5


def _raw_check(enc, rows, activation, expect_kernels):
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200._lib import ptr
    lib = _lib.load()
    dev = torch.device("cuda:0")
    desc, level = enc._plan.desc, 0
    theta, _ = enc._flat_params()
    lin = [(m.weight, m.bias) for m in enc.lgn_cg.mlp_levels[level].linear]
    nin, width = lin[0][0].shape[1], lin[0][0].shape[0]
    torch.manual_seed(rows + width)
    x = torch.randn(rows, nin, dtype=torch.float64, device=dev) * 2
    g_y = torch.randn(rows, nin, dtype=torch.float64, device=dev)
    wpack = torch.empty(lib.lgae_mlp_pack_doubles(C.byref(desc), level), dtype=torch.float64, device=dev)
    acts = torch.empty(len(lin) - 1, rows, 8 * ((width + 7) // 8), dtype=torch.float64, device=dev)
    y = torch.empty(rows, nin, dtype=torch.float64, device=dev)
    g_x = torch.empty_like(x)
    gtheta = torch.zeros_like(theta)
    partials = torch.empty(lib.lgae_partials_doubles(C.byref(desc), 1), dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def run():
        assert lib.lgae_mlp_forward(C.byref(desc), level, ptr(theta), ptr(x), rows, ptr(wpack), ptr(acts), ptr(y), st) == 0
        assert lib.lgae_mlp_backward(C.byref(desc), level, ptr(theta), ptr(x), rows, ptr(wpack), ptr(acts), ptr(g_y), ptr(g_x), ptr(gtheta),
                                     ptr(partials), st) == 0
        torch.cuda.synchronize()

    names = _lib.kernel_timings(run)
    fwd, bwd = expect_kernels
    assert fwd in names and bwd in names, (expect_kernels, sorted(names))
    assert not ({"mlp_fwd", "mlp_fwd_streamed", "mlp_bwd", "mlp_bwd_streamed"} - {fwd, bwd}) & set(names), sorted(names)
    g1 = gtheta.clone()
    gtheta.zero_()
    run()
    assert torch.equal(gtheta, g1)   # deterministic

    xr = x.detach().clone().requires_grad_(True)
    params = [(w.detach().clone().requires_grad_(True), b.detach().clone().requires_grad_(True)) for w, b in lin]
    h = xr
    for w, b in params[:-1]:
        h = ORACLE_ACTS[activation](F.linear(h, w, b))
    yr = F.linear(h, *params[-1])
    yr.backward(g_y)
    assert rel_err(y, yr.detach()) < 1e-10
    assert rel_err(g_x, xr.grad) < 1e-10
    names = [n for n, _ in enc.named_parameters() if n.startswith(f"lgn_cg.mlp_levels.{level}.linear.")]
    views = enc._plan.views(gtheta)
    ref = {f"lgn_cg.mlp_levels.{level}.linear.{i}.{'weight' if j == 0 else 'bias'}": t.grad
           for i, pair in enumerate(params) for j, t in enumerate(pair)}
    assert sorted(names) == sorted(ref)
    gmax = max(g.abs().max().item() for g in ref.values())
    for n in names:
        err = (views[n] - ref[n]).abs().max().item()
        assert err <= 1e-10 * max(ref[n].abs().max().item(), 1e-4 * gmax), (n, err)
    # the rest of theta's gradient stays zero
    mask = torch.ones_like(gtheta, dtype=torch.bool)
    for n in names:
        off, cnt, _ = enc._plan.offsets[n]
        mask[off:off + cnt] = False
    assert not gtheta[mask].any()


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [1, 21, "chunks"])
@pytest.mark.parametrize("depth", [1, 6])
@pytest.mark.parametrize("tiling", sorted(TILINGS))
def test_raw_mlp_matches_autograd(tiling, depth, rows):
    """lgae_mlp_forward / lgae_mlp_backward at every tiling of the streamed range against torch fp64 autograd, at 1 and 21 rows
    and at 32 * SMs * 3 + 5 rows (several 32-row chunks per CTA of the adjoint, a partial last group); the kernels that ran are
    the ones the selection rule names."""
    ntw, nti = tiling
    enc = _one_level(ntw, nti, depth, torch.device("cuda:0"))
    rows = _raw_rows(3) if rows == "chunks" else rows
    _raw_check(enc, rows, "leakyrelu", _kernel_names(ntw, nti, depth + 1))


@pytest.mark.gpu
@pytest.mark.parametrize("tiling,depth", [((8, 2), 6), ((9, 2), 5), ((9, 2), 6), ((9, 2), 7)])
def test_raw_mlp_mixed_families(tiling, depth):
    """Tilings with a resident instance past its adjoint's shared memory: resident forward and streamed adjoint, and at (9, 2)
    depth 7 both streamed."""
    ntw, nti = tiling
    expect = _kernel_names(ntw, nti, depth + 1)
    assert expect[1] == "mlp_bwd_streamed" and (expect[0] == "mlp_fwd_streamed") == (depth == 7)
    _raw_check(_one_level(ntw, nti, depth, torch.device("cuda:0")), _raw_rows(2), "leakyrelu", expect)


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ACTS)
def test_raw_mlp_activations_at_width_96(activation):
    enc = _one_level(12, 2, 3, torch.device("cuda:0"), activation)
    _raw_check(enc, _raw_rows(1), activation, ("mlp_fwd_streamed", "mlp_bwd_streamed"))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: modules and training steps against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_module_and_train_step_match_oracle(name, fused_only):
    """Module API + autograd, then FusedTrainStep (CUDA graph, captured and replayed), against one oracle step; two step runs give
    bit-identical gradients."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = CASES[name]
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 1e-8)
    batch = {k: v.to(dev) for k, v in batch_cpu.items() if k in ("p4", "labels")}
    latent = enc(batch)
    recon = dec(latent)
    loss = fused.chamfer_loss(recon, batch["p4"], "sum") + 1e-8 * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    lat = {key: latent[key].detach() for key in ((0, 0), (1, 1))}
    _assert_forward(name, lat, recon.detach(), loss.item(), ref_latent, ref_recon, ref_loss.item())
    _assert_grads(name, models, _grads(models), ref_grads)

    step = FusedTrainStep(enc, dec, cfg["batch"], l1_lambda=1e-8, normalize=False, use_labels=cfg["pad"], use_graph=True, get_real="sum")
    g_runs = []
    for _ in range(3):   # capture, then two replays
        l_step = step.step(batch["p4"], batch.get("labels")).item()
        torch.cuda.synchronize()
        g_runs.append(step.g_all.clone())
    _assert_forward(name + "/step", {(0, 0): step.latent00, (1, 1): step.latent11}, step.recon, l_step, ref_latent, ref_recon, ref_loss.item())
    _assert_grads(name + "/step", models, _grads(models), ref_grads)
    assert torch.equal(g_runs[1], g_runs[2]) and torch.equal(g_runs[0], g_runs[1]), name


@pytest.mark.gpu
def test_batch_past_the_persistent_grid(fused_only):
    """Batch 4 * SMs + 37 at width 50: many rows per CTA in both MLP directions."""
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.train import FusedTrainStep
    from tests.test_fused_coverage_gpu import cap_batch
    cfg = dict(CASES["c5_w50"], n=8, mlp_depth=1, pad=True)
    dev = torch.device("cuda:0")
    B = cap_batch(int(_lib.load().lgae_device_sm_count()))
    enc, dec = _build(cfg, dev)
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, B)
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 0.0)
    step = FusedTrainStep(enc, dec, B, l1_lambda=0.0, normalize=False, use_labels=True, use_graph=True, get_real="sum")
    for _ in range(2):
        loss = step.step(batch_cpu["p4"].to(dev), batch_cpu["labels"].to(dev)).item()
    torch.cuda.synchronize()
    _assert_forward("cap", {(0, 0): step.latent00, (1, 1): step.latent11}, step.recon, loss, ref_latent, ref_recon, ref_loss.item())
    _assert_grads("cap", models, _grads(models), ref_grads)


TILED_CFG = dict(seed=74, batch=2, n=40, num_basis_fn=3, enc_channels=[2, 6, 5], dec_channels=[5, 6, 3], tau_s=1, tau_v=2,
                 map_to_latent="min&max", mlp_depth=2, mlp_width=8, pad=True)   # widths 96 / 80 / 48


@pytest.mark.gpu
def test_tiled_train_step_at_40_particles(fused_only):
    from lgn_autoencoder_b200.train import FusedTrainStep
    cfg = TILED_CFG
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 1e-8)
    step = FusedTrainStep(enc, dec, cfg["batch"], l1_lambda=1e-8, normalize=False, use_labels=True, use_graph=True, get_real="sum",
                          adjoint="tiled")
    for _ in range(2):
        loss = step.step(batch_cpu["p4"].to(dev), batch_cpu["labels"].to(dev)).item()
    torch.cuda.synchronize()
    _assert_forward("tiled", {(0, 0): step.latent00, (1, 1): step.latent11}, step.recon, loss, ref_latent, ref_recon, ref_loss.item())
    _assert_grads("tiled", models, _grads(models), ref_grads)


@pytest.mark.gpu
def test_inference_past_32_particles_matches_module(fused_only):
    from lgn_autoencoder_b200.train import FusedInference
    cfg = dict(TILED_CFG, n=70, batch=3)
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    batch = {k: v.to(dev) for k, v in _jets(cfg, cfg["batch"]).items() if k in ("p4", "labels")}
    with torch.no_grad():
        latent = enc(batch)
        recon = dec(latent)
    inf = FusedInference(enc, dec, cfg["batch"], normalize=False, use_labels=True, get_real="sum")
    for _ in range(2):
        inf.score(batch["p4"], batch["labels"])
    torch.cuda.synchronize()
    assert rel_err(inf.recon, recon) < 1e-10
    assert rel_err(inf.latent11, latent[(1, 1)].reshape(inf.latent11.shape)) < 1e-10


@pytest.mark.gpu
def test_p4_grad_matches_oracle(fused_only, zero_mass_rule):
    cfg = CASES["cfg4_shape"]
    enc, dec = _build(cfg, torch.device("cuda:0"))
    batch = {k: v for k, v in _jets(cfg, cfg["batch"]).items() if k in ("p4", "labels")}
    g_p4, grads = _module_run(enc, dec, batch, "sum", True)
    _, grads_ref = _module_run(enc, dec, batch, "sum", False)
    err = rel_err(g_p4, _oracle_p4_grad(enc, dec, cfg, batch, "sum"))
    assert err <= 1e-10, err
    for k in grads:
        assert torch.equal(grads[k], grads_ref[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("activation", ACTS)
def test_activations_through_the_module(activation, fused_only, oracle_activation):
    from lgn_autoencoder_b200 import fused
    oracle_activation(activation)
    cfg = CASES["c5_w50"]
    dev = torch.device("cuda:0")
    enc, dec = _build(dict(cfg, mlp_width=9), dev, activation)   # widths 90 (ntw 12) and 36
    models = {"enc": enc, "dec": dec}
    batch_cpu = _jets(cfg, cfg["batch"])
    ref_loss, ref_latent, ref_recon, ref_grads = _oracle_step(enc, dec, cfg, batch_cpu, 1e-8)
    batch = {k: v.to(dev) for k, v in batch_cpu.items() if k in ("p4", "labels")}
    latent = enc(batch)
    recon = dec(latent)
    loss = fused.chamfer_loss(recon, batch["p4"], "sum") + 1e-8 * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    lat = {key: latent[key].detach() for key in ((0, 0), (1, 1))}
    _assert_forward(activation, lat, recon.detach(), loss.item(), ref_latent, ref_recon, ref_loss.item())
    _assert_grads(activation, models, _grads(models), ref_grads)


# launches of one eager cfg-1 training step (bench.py's model, 512 jets), as the parent commit of the streamed kernels made them
CFG1_STEP_LAUNCHES = 35


@pytest.mark.gpu
def test_step_kernel_names():
    """Per-kernel names of one eager step: cfg-1 launches no streamed kernel and as many kernels as before the streamed kernels
    existed; the wide model launches both streamed kernels."""
    from bench import build_models, synthetic_jets
    from lgn_autoencoder_b200 import _lib
    from lgn_autoencoder_b200.train import FusedTrainStep
    dev = torch.device("cuda:0")

    def names(enc, dec, p4):
        step = FusedTrainStep(enc, dec, p4.shape[0], l1_lambda=1e-8, normalize=True, use_labels=False, use_graph=False, get_real="sum")
        step.step(p4)
        torch.cuda.synchronize()
        return _lib.kernel_timings(lambda: (step.step(p4), torch.cuda.synchronize()))

    enc, dec = build_models(dev)
    cfg1 = names(enc, dec, synthetic_jets(512, 30, seed=3).to(dev))
    assert not [k for k in cfg1 if k.endswith("_streamed")], sorted(cfg1)
    assert "mlp_fwd" in cfg1 and "mlp_bwd" in cfg1
    assert sum(n for n, _ in cfg1.values()) == CFG1_STEP_LAUNCHES, cfg1
    cfg = dict(CASES["cfg4_shape"], mlp_depth=6)
    enc, dec = _build(cfg, dev)
    wide = names(enc, dec, _jets(cfg, 4)["p4"].to(dev))
    assert "mlp_fwd_streamed" in wide and "mlp_bwd_streamed" in wide, sorted(wide)
