"""The fused maxdim-3 forward (csrc/lgae_md3.cu): generated CG tables and piece order, C ABI size queries and eligibility on the
CPU; on the GPU, forward-only module calls, covariance outputs, FusedInference, equivariance, determinism and routing against
the golden vectors of the reference and the oracle."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from tests.helpers import load_golden, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------------------------------------------------------------------------
# CPU: tables and piece order
# ------------------------------------------------------------------------------------------------------------------


def test_generated_tables_match_cgdict():
    """The committed header is what tools/gen_md3_tables.py writes from CGDict(maxdim=3) today."""
    import runpy
    gen = runpy.run_path(os.path.join(ROOT, "tools", "gen_md3_tables.py"))
    with open(gen["HEADER"]) as f:
        assert f.read() == gen["render"]()


def test_terms_are_the_cg_coefficients():
    """Every non-zero CG coefficient of every (pair, output) piece appears once in the term lists, with its value."""
    from lgn_autoencoder_b200 import md3_layout as M
    from lgn_autoencoder_b200.cg_lib import CGDict
    cg = CGDict(maxdim=3)
    pieces, first, ranges, terms, _ = M.tables(cg)
    for p, (kind, r1, r2, t) in enumerate(pieces):
        if kind == M.KIND_NODE:
            assert all(ranges[first[p] + m] == ranges[first[p] + m + 1] for m in range(M.DIM[t]))
            continue
        mat = cg[(r1, r2)][t].numpy()
        rebuilt = np.zeros_like(mat)
        d2 = M.DIM[r2]
        for m in range(M.DIM[t]):
            for x, y, c in terms[ranges[first[p] + m]:ranges[first[p] + m + 1]]:
                if kind == M.KIND_SQ:
                    a, b = x - M.COMP_OFFSET[r1], y - M.COMP_OFFSET[r2]
                elif kind == M.KIND_AG1:
                    a, b = x // 4 - M.COMP_OFFSET[r1], x % 4
                else:
                    a, b = x - M.COMP_OFFSET[r1], 0
                rebuilt[m, a * d2 + b] += c
        assert np.abs(rebuilt - mat).max() <= M.COEF_EPS, (kind, r1, r2, t)


def _rand_rep(keys, shape, gen):
    return {k: torch.randn((2,) + shape + ((k[0] + 1) * (k[1] + 1),), generator=gen, dtype=torch.float64) for k in keys}


def _level_from_tables(variant, node, r0, r1, y, mix_w, cout):
    """One level evaluated the way the kernels do: neighbour sums S0 / T, then the pieces of the generated tables folded into the
    mix columns.  node: planar parts (2,B,N,C,d); r0, r1 (2,B,N,N,C) radial weights; y (2,B,N,N,4) edge vectors."""
    from lgn_autoencoder_b200 import md3_layout as M
    from lgn_autoencoder_b200.cg_lib import CGDict
    cg = CGDict(maxdim=3)
    pieces, first, ranges, terms, var_blocks = M.tables(cg)
    cx = lambda t: torch.complex(t[0], t[1])
    some = next(iter(node.values()))
    b, n, c = some.shape[1], some.shape[2], some.shape[3]
    z = torch.zeros((b, n, c, M.N_COMP), dtype=torch.complex128)
    for k, v in node.items():
        z[..., M.COMP_OFFSET[k]:M.COMP_OFFSET[k] + M.DIM[k]] = cx(v)
    R0, R1, Y = cx(r0), cx(r1), cx(y)
    S0 = torch.einsum("bijc,bjca->bica", R0, z)
    T = torch.einsum("bijc,bjca,bijd->bicad", R1, z, Y).reshape(b, n, c, 80)
    out = {}
    for t in M.IRREPS:
        cols = []
        for pid in var_blocks[variant][t]:
            kind = pieces[pid][0]
            vals = []
            for m in range(M.DIM[t]):
                if kind == M.KIND_NODE:
                    vals.append(z[..., M.COMP_OFFSET[t] + m])
                    continue
                acc = torch.zeros((b, n, c), dtype=torch.complex128)
                for x, yy, coef in terms[ranges[first[pid] + m]:ranges[first[pid] + m + 1]]:
                    if kind == M.KIND_SQ:
                        acc = acc + coef * z[..., x] * z[..., yy]
                    elif kind == M.KIND_AG1:
                        acc = acc + coef * T[..., x]
                    else:
                        acc = acc + coef * S0[..., x]
                if kind == M.KIND_AG0:
                    acc = acc * (1 + 1j)
                vals.append(acc)
            cols.append(torch.stack(vals, -1))          # (b, n, c, d)
        cat = torch.cat(cols, dim=2)                     # (b, n, ncols * c, d)
        w = cx(mix_w[t])
        o = torch.einsum("ok,bnkd->bnod", w, cat)
        out[t] = torch.stack([o.real, o.imag])
    return out


@pytest.mark.parametrize("variant", ["level0", "mlp", "nomlp"])
def test_piece_order_matches_composite(variant):
    """Pieces, columns and CG terms of the generated tables reproduce the oracle's node_level (cg_product / cat_reps / MixReps) on
    random node features, edges and mix weights, at level 0 and at later levels with either node key order."""
    from lgn_autoencoder_b200 import md3_layout as M
    from oracle import lgae_oracle as orc
    gen = torch.Generator().manual_seed(11)
    b, n, c, cout = 2, 4, 3, 2
    order = M.node_order(variant)
    node = _rand_rep(order, (b, n, c), gen)
    r0 = torch.randn((2, b, n, n, c), generator=gen, dtype=torch.float64)
    r1 = torch.randn((2, b, n, n, c), generator=gen, dtype=torch.float64)
    y = torch.randn((2, b, n, n, 4), generator=gen, dtype=torch.float64)
    cols = M.mix_columns(variant)
    mix_w = {t: torch.randn((2, cout, cols[t] * c), generator=gen, dtype=torch.float64) for t in M.IRREPS}
    one_pi = torch.ones((2, b, n, n, c, 1), dtype=torch.float64)          # zonal (0,0) of a pair: 1 + i
    edge = {(0, 0): orc.mul_zscalar_zirrep(r0, one_pi), (1, 1): orc.mul_zscalar_zirrep(r1, y.unsqueeze(-2).expand(2, b, n, n, c, 4))}
    ref = orc.node_level(orc.cg_table(3), node, edge, mix_w, 3)
    mine = _level_from_tables(variant, node, r0, r1, y, mix_w, cout)
    assert list(ref.keys()) == M.set_order(M.IRREPS)
    for t in M.IRREPS:
        assert rel_err(mine[t], ref[t]) < 1e-12, (variant, t, rel_err(mine[t], ref[t]))


def test_node_orders_match_the_modules():
    """The node key orders the kernels know are the ones the composite's modules produce."""
    from lgn_autoencoder_b200 import md3_layout as M
    from lgn_autoencoder_b200.models import LGNEncoder
    for mlp in (True, False):
        enc = LGNEncoder(num_input_particles=4, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=1, tau_latent_vectors=1,
                         maxdim=[3], num_basis_fn=4, num_channels=[2, 2, 2], max_zf=[1], weight_init="randn", level_gain=[1.0],
                         mlp=mlp, mlp_depth=1, mlp_width=2, map_to_latent="mean", device="cpu")
        assert list(enc.input_func_node.weights.keys()) == M.node_order("level0")
        mixed = list(enc.lgn_cg.node_levels[0].cat_mix.mix_reps.weights.keys())
        if mlp:
            mixed = [k for k in mixed if k != (0, 0)] + [(0, 0)]
        assert mixed == M.node_order("mlp" if mlp else "nomlp")
        for lvl, variant in zip(enc.lgn_cg.node_levels, ("level0", "mlp" if mlp else "nomlp")):
            cols = M.mix_columns(variant)
            assert dict(lvl.cat_mix.cat_reps.tau.items()) == {t: cols[t] * 2 for t in M.IRREPS}


# ------------------------------------------------------------------------------------------------------------------
# CPU: C ABI size queries and eligibility
# ------------------------------------------------------------------------------------------------------------------
def _plans(maxdim, n=30, enc_channels=(6, 6, 8, 8, 8), dec_channels=(8, 8, 6, 6, 6), mlp=True, mode="mix"):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    common = dict(maxdim=[maxdim], num_basis_fn=10, max_zf=[1], weight_init="randn", level_gain=[1.0], mlp=mlp, mlp_depth=6, mlp_width=6,
                  device="cpu")
    enc = LGNEncoder(num_input_particles=n, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=1, tau_latent_vectors=8,
                     num_channels=list(enc_channels), map_to_latent=mode, **common)
    dec = LGNDecoder(tau_latent_scalars=1, tau_latent_vectors=8, num_output_particles=n, tau_output_scalars=1, tau_output_vectors=1,
                     num_channels=list(dec_channels), cg_dict=enc.cg_dict, **common)
    return enc, dec


def test_size_queries():
    """maxdim 3: a workspace, no backward, no training step; maxdim 1 and 4 refused; maxdim 0 and 2 are the same descriptor."""
    from lgn_autoencoder_b200 import _lib
    lib = _lib.load()
    for n in (30, 150):
        enc, dec = _plans(3, n=n)
        de, dd = enc._plan.desc, dec._plan.desc
        assert de.maxdim == 3 and dd.maxdim == 3
        for d in (de, dd):
            assert lib.lgae_workspace_doubles(C.byref(d), 16) > 0
            assert lib.lgae_workspace_offset(C.byref(d), 16, 9, 1) > 0          # (2,0) | (0,2) | (2,2) parts
            assert lib.lgae_workspace_offset(C.byref(d), 16, 9, 0) == -1         # level 0: (0,0), (1,1) only
            assert lib.lgae_workspace_offset(C.byref(d), 16, 4, 0) == -1         # no saved neighbour sums
            assert lib.lgae_partials_doubles(C.byref(d), 16) == -2
            assert lib.lgae_backward_tiled_scratch_doubles(C.byref(d), 16) == -2
        assert lib.lgae_encoder_input_grad_scratch_doubles(C.byref(de), 16) == -2
        assert lib.lgae_train_step_partials_doubles(C.byref(de), C.byref(dd), 16) == -2
        assert lib.lgae_train_step_tiled_scratch_doubles(C.byref(de), C.byref(dd), 16) == -2
        for bad in (1, 4, -1):
            for d in (de, dd):
                d.maxdim = bad
                assert lib.lgae_workspace_doubles(C.byref(d), 16) == -1
                d.maxdim = 3
    for n in (30, 150):
        enc, dec = _plans(2, n=n, enc_channels=(3, 3, 4), dec_channels=(4, 3, 3), mode="mean")
        de, dd = enc._plan.desc, dec._plan.desc
        queries = lambda: ([lib.lgae_workspace_doubles(C.byref(d), 16) for d in (de, dd)]
                           + [lib.lgae_workspace_offset(C.byref(d), 16, k, l) for d in (de, dd) for k in range(10) for l in range(3)]
                           + [lib.lgae_partials_doubles(C.byref(d), 16) for d in (de, dd)]
                           + [lib.lgae_backward_tiled_scratch_doubles(C.byref(d), 16) for d in (de, dd)]
                           + [lib.lgae_encoder_input_grad_scratch_doubles(C.byref(de), 16),
                              lib.lgae_train_step_partials_doubles(C.byref(de), C.byref(dd), 16),
                              lib.lgae_train_step_tiled_scratch_doubles(C.byref(de), C.byref(dd), 16)])
        assert de.maxdim == 2 and dd.maxdim == 2
        two = queries()
        de.maxdim = dd.maxdim = 0
        assert queries() == two


def test_eligibility():
    """cfg-4 (enc 6-6-8-8 / dec 8-8-6-6, 'mix', MLP 6 x 6) runs forward-only calls fused and trains on the composite; a mixed
    per-level maxdim runs neither fused."""
    enc, dec = _plans(3)
    for m in (enc, dec):
        assert not m.fused and m.fused_forward
        assert m._fused_reason.startswith("maxdim")
        assert m._forward_reason is None
    from lgn_autoencoder_b200.models import LGNEncoder
    mixed = LGNEncoder(num_input_particles=5, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=1, tau_latent_vectors=1,
                       maxdim=[2, 3, 3], num_basis_fn=4, num_channels=[2, 2, 2, 2], max_zf=[1], weight_init="randn", level_gain=[1.0],
                       mlp=True, mlp_depth=1, mlp_width=2, map_to_latent="mean", device="cpu")
    assert not mixed.fused and not mixed.fused_forward
    enc2, dec2 = _plans(2, enc_channels=(3, 3), dec_channels=(3, 3), mode="mean")
    assert enc2.fused and enc2.fused_forward and dec2.fused and dec2.fused_forward


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
ORACLE_ACTS = {
    "leakyrelu": lambda x: torch.nn.functional.leaky_relu(x, 0.01),
    "elu": torch.nn.functional.elu,
    "tanh": torch.tanh,
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
                x = act(torch.nn.functional.linear(x, w, b))
            w, b = linears[-1]
            x = torch.nn.functional.linear(x, w, b)
            rep[(0, 0)] = x.view(s[1:] + (2,)).permute(3, 0, 1, 2).unsqueeze(-1)
            return rep

        monkeypatch.setattr(orc, "cgmlp", cgmlp)

    return use


def _build(cfg, dev):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg.get("seed", 0))
    common = dict(maxdim=[3], num_basis_fn=cfg.get("nb", 4), max_zf=[1], weight_init="randn", level_gain=[1.0],
                  activation=cfg.get("act", "leakyrelu"), mlp=cfg.get("mlp", True), mlp_depth=cfg.get("depth", 2), mlp_width=cfg.get("width", 2),
                  device=dev, dtype=torch.float64)
    mode = cfg.get("mode", "mean")
    ts, tv = cfg.get("tau_s", 1), cfg.get("tau_v", 2)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=ts, tau_latent_vectors=tv,
                     num_channels=cfg["enc"], map_to_latent=mode, scale=cfg.get("scale", 1.0), **common)
    mult = 2 if mode == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=ts * mult, tau_latent_vectors=tv * mult, num_output_particles=cfg["n"], tau_output_scalars=1,
                     tau_output_vectors=1, num_channels=cfg["dec"], cg_dict=enc.cg_dict, **common)
    assert enc.fused_forward and dec.fused_forward and not enc.fused and not dec.fused
    return enc, dec


def _jets(cfg, dev):
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(cfg["b"], cfg["n"], seed=cfg.get("seed", 0), pad=cfg.get("pad", False))
    return {k: v.to(dev) for k, v in data.items()}


def _oracle(enc, dec, cfg, data):
    from oracle import lgae_oracle as orc
    esd = {k: v.detach().cpu() for k, v in enc.state_dict().items()}
    dsd = {k: v.detach().cpu() for k, v in dec.state_dict().items()}
    ecfg = dict(num_channels=cfg["enc"], maxdim=[3], max_zf=[1], map_to_latent=cfg.get("mode", "mean"), scale=cfg.get("scale", 1.0))
    dcfg = dict(num_channels=cfg["dec"], maxdim=[3], max_zf=[1])
    cpu = {k: v.cpu() for k, v in data.items()}
    lat, nodes = orc.encoder_forward(esd, ecfg, cpu, covariance_test=True)
    if cfg.get("mode", "mean") == "sum":
        return lat, None, nodes
    recon = orc.decoder_forward(dsd, dcfg, lat)
    return lat, recon, nodes


RANDOM_CASES = {
    "mix_c1_3_8_5": dict(seed=1, b=3, n=5, enc=[1, 3, 8, 5], dec=[5, 8, 3, 1], mode="mix", tau_v=3),
    "mean_n1": dict(seed=2, b=4, n=1, enc=[2, 3], dec=[3, 2], mode="mean"),
    "sum_n30": dict(seed=3, b=2, n=30, enc=[3, 4, 2], dec=[2, 3], mode="sum"),
    "min_n32_pad": dict(seed=4, b=3, n=32, enc=[2, 3, 3], dec=[3, 2], mode="min", pad=True),
    "max_n33_pad": dict(seed=5, b=2, n=33, enc=[3, 2], dec=[2, 4, 3], mode="max", pad=True),
    "minmax_n64": dict(seed=6, b=2, n=64, enc=[2, 2], dec=[2, 2], mode="min&max", scale=2.5),
    "mean_n150_pad": dict(seed=7, b=2, n=150, enc=[2, 3], dec=[3, 2], mode="mean", pad=True, nb=10),
    "nomlp": dict(seed=8, b=2, n=7, enc=[3, 4, 3], dec=[3, 4, 2], mode="mean", mlp=False),
    "wide_mlp_elu": dict(seed=9, b=2, n=6, enc=[4, 8, 7], dec=[7, 8, 4], mode="mix", width=6, act="elu"),   # widths 96, 84
    "narrow_tanh": dict(seed=10, b=2, n=9, enc=[3, 5], dec=[5, 3], mode="mean", width=3, depth=3, act="tanh"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RANDOM_CASES))
def test_forward_matches_oracle(name, fused_only, oracle_activation):
    """No-grad module calls on the fused maxdim-3 kernels against the oracle: latents, reconstruction and every covariance node."""
    cfg = RANDOM_CASES[name]
    oracle_activation(cfg.get("act", "leakyrelu"))
    dev = torch.device("cuda:0")
    enc, dec = _build(cfg, dev)
    data = _jets(cfg, dev)
    ref_lat, ref_recon, ref_nodes = _oracle(enc, dec, cfg, data)
    with torch.no_grad():
        lat, nodes = enc(data, covariance_test=True)
        for key in ((0, 0), (1, 1)):
            assert rel_err(lat[key], ref_lat[key]) < 1e-10, (name, key, rel_err(lat[key], ref_lat[key]))
        assert len(nodes) == len(ref_nodes)
        for i, (mine, ref) in enumerate(zip(nodes, ref_nodes)):
            assert list(mine.keys()) == list(ref.keys()), (i, list(mine.keys()), list(ref.keys()))
            # relative to the node's largest part: with one particle the (2,0) / (0,2) parts are the antisymmetric self product
            # of a vector, zero up to rounding in both implementations
            scale = max(v.abs().max().item() for v in ref.values())
            for key, val in ref.items():
                err = (mine[key].cpu() - val).abs().max().item() / scale
                assert err < 1e-10, (name, i, key, err)
        if ref_recon is not None:
            recon = dec(lat)
            assert rel_err(recon, ref_recon) < 1e-10, (name, rel_err(recon, ref_recon))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["md3_mix_n5", "cfg4_b2"])
def test_golden_no_grad(name, fused_only):
    """The reference's golden vectors, forward-only, on the fused maxdim-3 kernels: latents, reconstruction, every covariance
    node GVec in the same part order."""
    from tests.test_models_gpu import load
    g, enc, dec, batch = load(name, torch.device("cuda:0"))
    assert enc.fused_forward and dec.fused_forward
    with torch.no_grad():
        latent = enc(batch)
        recon = dec(latent)
        for key, val in g["latent"].items():
            assert rel_err(latent[eval(key)], val) < 1e-10, ("latent", key, rel_err(latent[eval(key)], val))
        assert rel_err(recon, g["recons"]) < 1e-10, rel_err(recon, g["recons"])
        lat2, nodes = enc(batch, covariance_test=True)
        gen, nodes_all = dec(lat2, covariance_test=True, nodes_all=nodes)
    assert len(nodes_all) == len(g["nodes_all"])
    for i, (mine, ref) in enumerate(zip(nodes_all, g["nodes_all"])):
        assert [str(k) for k in mine.keys()] == list(ref.keys()), (i, list(mine.keys()), list(ref.keys()))
        for key, val in ref.items():
            assert rel_err(mine[eval(key)], val) < 1e-10, (i, key, rel_err(mine[eval(key)], val))


@pytest.mark.gpu
def test_batch_past_persistent_grid_and_determinism(fused_only):
    """A batch of more jets than CTAs fit on the device at once; repeated calls bit-identical; one jet alone bit-identical to the
    same jet inside the batch."""
    from lgn_autoencoder_b200 import _lib
    dev = torch.device("cuda:0")
    cfg = dict(seed=12, b=4 * _lib.load().lgae_device_sm_count() + 3, n=12, enc=[3, 4, 3], dec=[3, 4, 3], mode="mix", pad=True)
    enc, dec = _build(cfg, dev)
    data = _jets(cfg, dev)
    with torch.no_grad():
        lat = enc(data)
        recon = dec(lat)
        lat_b = enc(data)
        assert all(torch.equal(lat[k], lat_b[k]) for k in lat.keys())
        assert torch.equal(dec(lat_b), recon)
        for j in (0, cfg["b"] - 1):
            one = {k: v[j:j + 1] for k, v in data.items()}
            l1 = enc(one)
            for k in l1.keys():
                assert torch.equal(l1[k], lat[k][:, j:j + 1]), k
            assert torch.equal(dec(l1), recon[:, j:j + 1])
    sub = {k: v[:3].cpu() for k, v in data.items()}
    ref_lat, ref_recon, _ = _oracle(enc, dec, dict(cfg, b=3), sub)
    assert rel_err(recon[:, :3], ref_recon) < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("n", [30, 150])
def test_fused_inference(n):
    """FusedInference on a maxdim-3 model: scores against the per-jet chamfer of the composite's reconstruction, graph replay
    bit-identical to eager, all_scores against the oracle."""
    from lgn_autoencoder_b200.train import FusedInference
    from oracle import lgae_oracle as orc
    dev = torch.device("cuda:0")
    cfg = dict(seed=13, b=5, n=n, enc=[3, 4, 3], dec=[3, 4, 3], mode="mix", tau_v=2, pad=True, nb=6)
    enc, dec = _build(cfg, dev)
    data = _jets(cfg, dev)
    p4 = data["p4"]
    graph = FusedInference(enc, dec, cfg["b"], get_real="sum", use_labels=True)
    eager = FusedInference(enc, dec, cfg["b"], get_real="sum", use_labels=True, use_graph=False)
    s_graph = graph.score(p4, data["labels"]).clone()
    s_graph2 = graph.score(p4, data["labels"]).clone()
    s_eager = eager.score(p4, data["labels"]).clone()
    assert torch.equal(s_graph, s_eager) and torch.equal(s_graph, s_graph2)
    pn, _ = orc.normalize_p4_overall_max(p4.cpu())
    with torch.enable_grad():   # the composite: a grad-enabled call of a maxdim-3 model
        lat = enc({"p4": pn.to(dev), "labels": data["labels"]})
        recon = dec(lat).detach().cpu()
    ref = torch.stack([orc.chamfer_loss(orc.get_real(recon[:, j:j + 1], "sum"), pn[j:j + 1]) for j in range(cfg["b"])])
    assert rel_err(s_eager, ref) < 1e-10, rel_err(s_eager, ref)
    scores = graph.all_scores()
    ref_scores = orc.anomaly_scores_cartesian(orc.get_real(graph.recon.cpu(), "sum"), pn)
    for k, v in ref_scores.items():
        # the Minkowski scores are differences of squares: their error is measured on the Euclidean counterpart's scale
        scale = ref_scores[k.replace("lorentz", "cartesian")].abs().max().item()
        assert (scores[k].cpu() - v).abs().max().item() < 1e-10 * scale, k


@pytest.mark.gpu
def test_equivariance_no_worse_than_composite():
    """The equivariance harness (boosts and rotations, under no_grad) on a small maxdim-3 model: the fused forward's deviations
    are at most 3x the composite's on the same jets and weights."""
    from lgn_autoencoder_b200.models.autotest import covariance_test
    dev = torch.device("cuda:0")
    cfg = dict(seed=14, b=2, n=6, enc=[2, 3], dec=[3, 2], mode="mean", pad=False)
    enc, dec = _build(cfg, dev)
    data = _jets(cfg, dev)
    data["p4"] = data["p4"] * 1e3     # the harness works in GeV
    results = {}
    with torch.no_grad():
        results["fused"] = [covariance_test(enc, dec, data, t) for t in ("boost", "rotation")]
        enc._forward_reason = dec._forward_reason = "the composite, for comparison"
        results["composite"] = [covariance_test(enc, dec, data, t) for t in ("boost", "rotation")]
    def flat(x):
        if torch.is_tensor(x):
            return [x.abs().max().item()]
        if isinstance(x, dict):
            return [v for k in sorted(x, key=str) for v in flat(x[k])]
        if isinstance(x, (list, tuple)):
            return [v for e in x for v in flat(e)]
        return [abs(float(x))]
    for t, (mine, ref) in enumerate(zip(results["fused"], results["composite"])):
        for key in mine:
            if key in ("gammas", "thetas"):
                continue
            a, b = flat(mine[key]), flat(ref[key])
            assert len(a) == len(b)
            for x, y in zip(a, b):
                assert x <= 3 * y + 1e-13, (t, key, x, y)


@pytest.mark.gpu
def test_routing():
    """Grad-enabled calls run the composite with matching gradients; no-grad calls launch only fused kernels; FusedTrainStep refuses."""
    from lgn_autoencoder_b200 import _lib, fused
    from lgn_autoencoder_b200.train import FusedTrainStep
    from tests.test_models_gpu import load
    from tests.helpers import assert_grads_close
    g, enc, dec, batch = load("md3_mix_n5", torch.device("cuda:0"))
    latent = enc(batch)
    recon = dec(latent)
    loss = fused.chamfer_loss(recon, batch["p4"], g["cfg"].get("get_real", "sum")) + 1e-8 * (enc.l1_norm() + dec.l1_norm())
    loss.backward()
    assert_grads_close({k: p.grad for k, p in dec.named_parameters()}, g["grads_dec"])
    assert_grads_close({k: p.grad for k, p in enc.named_parameters()}, g["grads_enc"])

    def run():
        with torch.no_grad():
            dec(enc(batch))
    run()
    names = _lib.kernel_timings(run)
    assert any(n.startswith("md3_") for n in names), names
    composite = {"cg_product", "cg_aggregate", "mix", "linear", "scalar_irrep", "radial_functions"}
    assert not [n for n in names if any(n.startswith(c) for c in composite)], names
    with pytest.raises(NotImplementedError):
        FusedTrainStep(enc, dec, batch["p4"].shape[0])
