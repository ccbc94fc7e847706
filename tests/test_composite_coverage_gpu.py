"""Coverage of the layer-level composite (csrc/lgae_cg.cu, csrc/lgae_layers.cu driven by layer_ops.py through autograd), the
path that trains every configuration the fused path refuses: maxdim 3, max_zf > 1, more than 8 channels, more than 16 radial
basis functions.

Three parts:

* No GPU: the host dispatch rules of the layer launchers, restated below with the lines they come from, and the case tables
  of the GPU tests.  ``test_case_tables_reach_every_branch`` fails if the tables stop reaching a branch, if a grid-capped
  launcher has no case past its cap on a 148-SM B200, or if the library gains a kernel instance (LGAE_KRON, LGAE_MULTI,
  LGAE_LIN, parsed from the sources) that no case launches.
* GPU: every layer op through the autograd functions the modules use, against a plain fp64 reference on the CPU (the
  oracle's restatement of the reference, or torch fp64 of the same op), outputs and the gradient of every input for a random
  cotangent.  Shapes are computed from the device's SM count, so the capped cases run past the cap on any part.
* GPU: models only the composite trains.  cfg-4 exactly as bench.py builds it, at batch 1024, against the fused maxdim-3
  forward (every jet), the oracle (a handful of jets, forward and parameter gradients) and the sum of 8-jet chunks; and small
  batches of max_zf = 2, 9-16 channels and 17-20 radial basis functions against the oracle.

Tolerances: 1e-12 relative (max-norm) where an output element is a sum of at most a few hundred products.  A reduction over
n >> 100 terms (weight gradients over all rows, parameter gradients of the radial functions over all edges) is checked
element-wise against the a-priori bound of a recursive fp64 sum, |got - ref| <= 2 n u sum|term| (u = 2^-53; both sides carry
such an error), see ``_assert_sum_close``."""
import os
import re

import pytest
import torch

from tests.helpers import assert_grads_close, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lgn_autoencoder_b200", "csrc")
TOL = 1e-12
U = 2.0 ** -53
B200_SMS = 148
KB = 1024

IRREPS3 = [(0, 0), (1, 1), (0, 2), (2, 0), (2, 2)]     # node irreps of a maxdim-3 model (D1T = 20)


def _dim(key):
    return (key[0] + 1) * (key[1] + 1)


# ---------------------------------------------------------------------------------------------------------------------
# instance lists and tuning constants, read from the sources
# ---------------------------------------------------------------------------------------------------------------------
def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _between(text, start, end):
    i = text.index(start)
    return text[i:text.index(end, i)]


def _define(name, macro):
    return int(re.search(r"#define\s+" + macro + r"\s+(\d+)", _source(name)).group(1))


def _instances(text, macro):
    return {tuple(int(v) for v in m) if len(m) > 1 else int(m[0])
            for m in (tuple(x for x in t if x) for t in re.findall(macro + r"\((\d+)(?:,\s*(\d+))?\)", text))}


def source_instances():
    cg, layers = _source("lgae_cg.cu"), _source("lgae_layers.cu")
    fwd = _between(cg, "int lgae_cg_product_forward(", "int lgae_cg_product_backward(")
    bwd = _between(cg, "int lgae_cg_product_backward(", "static int multi_fill(")
    mbwd = _between(cg, "int lgae_cg_aggregate_multi_backward(", "static int multi_fill(CgMultiArgs& p")
    mfwd = _between(cg, "int lgae_cg_aggregate_multi_forward(", "int64_t lgae_mix_partials_doubles(")
    return {
        "kron_fwd": {v for v in _instances(fwd, "LGAE_KRON") if isinstance(v, int)},
        "kron_edge": {v for v in _instances(bwd, "LGAE_KRON") if isinstance(v, int)},
        "kron_node": {v for v in _instances(bwd, "LGAE_KRON") if isinstance(v, tuple)},
        "multi_fwd": _instances(mfwd, "LGAE_MULTI"),
        "multi_edge": _instances(mbwd, "LGAE_MULTI"),
        "multi_node": {(int(a), int(b)) for a, b in re.findall(r"cg_agg_multi_bwd_node_kernel<(\d+),\s*(\d+)>", mbwd)},
        "lin": _instances(layers, "LGAE_LIN"),
        "agg_fwd_ib": _define("lgae_cg.cu", "LGAE_AGG_FWD_IB"),
        "agg_edge_ib": _define("lgae_cg.cu", "LGAE_AGG_EDGE_IB"),
        "rad_eb": _define("lgae_layers.cu", "LGAE_RAD_EB"),
        "rad_ctas": _define("lgae_layers.cu", "LGAE_RAD_CTAS"),
    }


# ---------------------------------------------------------------------------------------------------------------------
# dispatch rules, restated from the host code
# ---------------------------------------------------------------------------------------------------------------------
def grid_for(work, threads, sms):
    """lgae_cg.cu:968 and lgae_layers.cu:14: ceil(work / threads) CTAs, at most 8 per SM; the kernels grid-stride."""
    return max(1, min(-(-work // threads), 8 * sms))


def grid_stride_pass(work, threads, sms):
    """(CTAs, items one pass of the whole grid covers, items per CTA) of a grid_for launch."""
    g = grid_for(work, threads, sms)
    return g, g * threads, threads


def terms_doubles(n_terms, n_start):
    """lgae_cg.cu:68."""
    return n_terms + (3 * n_terms + n_start + 1) // 2


SMEM_MAX = 227 * KB   # dynamic shared memory one sm_100 CTA may opt in to (lgae_cg.cu CG_SMEM_MAX)


def cg_row_stride(n):
    """lgae_cg.cu:80."""
    return n | 1


def cg_tile(C, d1, d2, nj, fixed, bwd):
    """lgae_cg.cu cg_tile (:991-998): neighbour tile next to `fixed` bytes in 160 KB; the adjoint also caps it at 4 x 256 z1 items."""
    per_j = (cg_row_stride(C * d1) + cg_row_stride(C * d2)) * 16
    if fixed + per_j > 160 * KB:
        return 0, per_j
    jt = (160 * KB - fixed) // per_j
    if bwd:
        jt = min(jt, 4 * 256 // (C * d1))
    return min(jt, nj), per_j


def cg_pair_fwd(C, d1, d2, n_comp, n_terms, B, nj, kron, sms):
    """lgae_cg_product_forward (lgae_cg.cu:1006-1069) for one pair, kernel order (d2: the edge side).  Returns (kernel, dynamic
    shared memory, grid details): point-wise for nj = 0; when the node slab and one edge row block fit in 100 KB next to the
    term table, the whole-jet Kronecker kernel of its d2 if its K buffer fits too, else the whole-jet block kernel; otherwise the
    neighbour-split kernel, whose grid (B, split) strides over the particles i."""
    if nj == 0:
        return ("pointwise", terms_doubles(n_terms, n_comp + 1) * 8, None)
    assert C * n_comp <= 4 * 256                                     # :1028 (LGAE_E_UNSUPPORTED beyond)
    fixed0 = terms_doubles(n_terms, n_comp + 1) * 8
    z1b, rowb = nj * C * d1 * 16, nj * C * d2 * 16
    if fixed0 + z1b + rowb <= 100 * KB:                              # :1030-1056
        ib = min(max(1, 256 // (C * n_comp)), nj)
        while ib > 1 and fixed0 + z1b + ib * rowb > 100 * KB:
            ib -= 1
        nbytes, kb = fixed0 + z1b + ib * rowb, ib * C * d1 * d2 * 16
        if d2 in kron and nbytes + kb <= SMEM_MAX:
            return (f"kron{d2}", nbytes + kb, None)
        return ("block", nbytes, ("kron_too_big" if d2 in kron else None))
    jt, per_j = cg_tile(C, d1, d2, nj, fixed0, False)               # :1057-1068 (the grid: :1064-1067)
    assert jt >= 1
    split = max(1, min(-(-2 * sms // B), nj))
    return ("split", fixed0 + jt * per_j, dict(jt=jt, split=split, n=nj))


def cg_pair_bwd(C, d1, d2, n_comp, n_terms, nj, g1, g2, kron_edge, kron_node):
    """lgae_cg_product_backward (lgae_cg.cu:1071-1161): the launches for the node (g1) and edge (g2) gradients, each as
    (kernel, dynamic shared memory)."""
    terms = (terms_doubles(n_terms, d1 + 1) + terms_doubles(n_terms, d2 + 1)) * 8
    if nj == 0:
        return [("pointwise", terms)]
    assert C * d1 <= 4 * 256                                         # :1094
    out = []
    if g2:                                                           # :1095-1127 edge gradient alone
        ib = min(8, nj)
        nbytes = terms_doubles(n_terms, d2 + 1) * 8 + (nj * C * d1 + ib * C * n_comp) * 16
        if nbytes <= 100 * KB:
            kbytes = terms_doubles(n_terms, d1 + 1) * 8 + (nj * C * d1 + ib * C * n_comp + ib * C * d1 * d2) * 16
            if d2 in kron_edge and kbytes <= SMEM_MAX:
                out.append((f"edge_kron{d2}", kbytes))
            else:
                out.append(("edge_generic" if d2 not in kron_edge else "edge_generic_kron_too_big", nbytes))
            g2 = False
            if not g1:
                return out
    if not g2 and g1 and nj * C <= 2 * 256:                          # :1128-1152 node gradient, Kronecker form
        t1 = terms_doubles(n_terms, d1 + 1) * 8
        per_ib = nj * C * d2 * 16 + (C * n_comp + C * d1 * d2) * 16
        ib = min(4, nj)
        while ib > 1 and t1 + ib * per_ib > 100 * KB:
            ib -= 1
        if t1 + ib * per_ib <= 100 * KB and (d1, d2) in kron_node:
            return out + [(("node_kron", d1, d2), t1 + ib * per_ib)]
    fixed = terms + C * n_comp * 16                                  # :1153-1161
    jt, per_j = cg_tile(C, d1, d2, nj, fixed, True)
    assert jt >= 1
    return out + [("tiled", fixed + jt * per_j)]


def multi_fwd(C, nj, d1t, d2t, n_comp, n_terms, src):
    """lgae_cg_aggregate_multi_forward (lgae_cg.cu:1246-1271): (kernel, ib, dynamic shared memory) or 'fallback'
    (LGAE_E_UNSUPPORTED: layer_ops then launches the pairs one by one)."""
    fixed = n_terms * 8 + (2 * n_terms + 4 * n_comp + 2) * 4 + 16
    per_ib = (nj * C * d2t + C * d1t * d2t) * 16
    ib = min(src["agg_fwd_ib"], nj)
    while ib > 1 and fixed + ib * per_ib > 100 * KB:
        ib -= 1
    if fixed + ib * per_ib > 160 * KB or d2t not in src["multi_fwd"]:
        return "fallback"
    return (f"multi_fwd{d2t}", ib, fixed + ib * per_ib)


def multi_bwd(C, nj, d1t, d2t, n_comp, n_terms, want_node, want_edge, src):
    """lgae_cg_aggregate_multi_backward (lgae_cg.cu:1166-1218): the launches as (kernel, ib, dynamic shared memory), or
    'fallback' (every gradient then comes from the per-pair adjoint)."""
    ncell = d1t * d2t
    tabs = n_terms * 8 + (n_terms + ncell + 1 + 3 * n_comp) * 4 + 16
    if want_node and not ((d1t, d2t) in src["multi_node"] and nj * C <= 256):
        return "fallback"
    if want_edge and d2t not in src["multi_edge"]:
        return "fallback"
    out = []
    if want_edge:
        per_ib = (C * n_comp + C * ncell) * 16
        ib = min(src["agg_edge_ib"], nj)
        while ib > 1 and tabs + ib * per_ib > 100 * KB:
            ib -= 1
        if tabs + ib * per_ib > 160 * KB:
            return "fallback"
        out.append((f"multi_edge{d2t}", ib, tabs + ib * per_ib))
    if want_node:
        per_ib = (nj * C * d2t + C * n_comp + C * ncell) * 16
        ib = min(2, nj)
        while ib > 1 and tabs + ib * per_ib > 100 * KB:
            ib -= 1
        if tabs + ib * per_ib > 160 * KB:
            return "fallback"
        out.append((f"multi_node{d1t}", ib, tabs + ib * per_ib))
    return out


def node_ok(d1t, d2t, nj, C):
    """layer_ops._CGPairsFn.backward (layer_ops.py:249): the node gradients go to the one-launch adjoint only here."""
    return d2t == 5 and d1t in (5, 20) and nj * C <= 256


def cg_route(case, src, sms):
    """Every launch of one cg_product call and its adjoint (both operands' gradients), as layer_ops and the host code pick
    them: the python side (plan_pairs, plan_multi :172-185, node_ok) runs as is on CPU tensors of the right shapes.  Returns
    records (what, name, dynamic shared memory, details)."""
    from lgn_autoencoder_b200 import layer_ops
    cg = _cgdict()
    node, edge = case["node"], case["edge"]
    swap = case["swap"]
    rep1, rep2 = (edge, node) if swap else (node, edge)
    keys1, keys2 = list(rep1), list(rep2)
    agg = case["agg"]
    B, nj = (case["batch"][0], case["batch"][1]) if agg else (case["batch"][0], 0)
    top = max(max(k for k, _ in keys1) + max(k for k, _ in keys2), max(n for _, n in keys1) + max(n for _, n in keys2)) + 1
    max_dim = int(min(top, case["maxdim"]))
    pairs, out_keys, out_ch = layer_ops.plan_pairs(cg, keys1, keys2, [rep1[k] for k in keys1], [rep2[k] for k in keys2], max_dim, swap,
                                                   torch.device("cpu"))
    p1 = [torch.empty(2, 1, rep1[k], _dim(k)) for k in keys1]
    p2 = [torch.empty(2, 1, rep2[k], _dim(k)) for k in keys2]
    out = []
    mp = layer_ops.plan_multi(cg, pairs, p1, p2, out_keys, out_ch, swap) if agg else None
    fwd_multi = False
    if mp is not None:
        f = multi_fwd(mp.desc.channels, nj, mp.d1t, mp.d2t, mp.desc.n_comp, mp.desc.n_terms, src)
        fwd_multi = f != "fallback"
        out.append(("multi", f[0], f[2], f[1]) if fwd_multi else ("fallback", "fwd", 0, None))
    pair_bwd_node, pair_bwd_edge = True, True
    if fwd_multi:
        want_node = node_ok(mp.d1t, mp.d2t, nj, mp.desc.channels)
        out.append(("node_ok", want_node, 0, (mp.d1t, nj * mp.desc.channels)))
        b = multi_bwd(mp.desc.channels, nj, mp.d1t, mp.d2t, mp.desc.n_comp, mp.desc.n_terms, want_node, True, src)
        if b == "fallback":
            out.append(("fallback", "bwd", 0, None))
        else:
            out += [("multi", name, smem, ib) for name, ib, smem in b]
            pair_bwd_edge, pair_bwd_node = False, not want_node
    for pp in pairs:
        d = pp.desc
        if not fwd_multi:
            name, smem, info = cg_pair_fwd(d.channels, d.d1, d.d2, d.n_comp, d.n_terms, B, nj, src["kron_fwd"], sms)
            out.append(("fwd", name, smem, info))
            if name == "pointwise":
                out.append(("pt_work", "fwd", 0, B * d.channels * d.n_comp))
        if pair_bwd_node or pair_bwd_edge:
            for name, smem in cg_pair_bwd(d.channels, d.d1, d.d2, d.n_comp, d.n_terms, nj, pair_bwd_node, pair_bwd_edge, src["kron_edge"],
                                          src["kron_node"]):
                out.append(("bwd", name, smem, None))
                if name == "pointwise":
                    out.append(("pt_work", "bwd", 0, B * d.channels * (d.d1 + d.d2)))
    return out


def mix_route(rows, cin, cout, d, sms):
    """lgae_mix_forward / lgae_mix_backward (lgae_cg.cu:1273-1354): COV 4 / 8 / 16 (blocks of 16 output channels), co_blk of
    the weight gradient, its CTAs (rows_per_cta rows each, at most 4 per SM) and the grid_for launches."""
    cov = 4 if cout <= 4 else (8 if cout <= 8 else 16)
    ctas = max(1, min(rows, 4 * sms))
    rpc = -(-rows // ctas)
    return dict(cov=cov, co_blocks=-(-cout // 16) if cov == 16 else 1, co_blk=4 if cout <= 4 else 8, rows_per_cta=rpc,
                w_grid=-(-rows // rpc), fwd=grid_stride_pass(rows * d, 256, sms), bwd_x=grid_stride_pass(rows * cin * d, 256, sms))


def lin_route(rows, nin, nout, sms, lin_nt):
    """lgae_linear_forward / _backward (lgae_layers.cu:521-543, 639-700): MMA when both widths are <= 128 (bwd_w: n_in + 1), the
    tile width NT of launch_lin_mma (forward N = n_out, bwd_x N = n_in), lin_splits and the MMA grid."""
    def nt_of(n):
        nt = -(-n // 8)
        return min(v for v in sorted(lin_nt) if nt <= v or v == max(lin_nt))
    units = -(-rows // 16)
    mma_grid = max(1, min(-(-units // 8), sms))
    splits = max(1, min(-(-rows // 128), sms))
    return dict(fwd=("mma", nt_of(nout)) if nin <= 128 and nout <= 128 else ("fma",),
                bwd_x=("mma", nt_of(nin)) if nin <= 128 and nout <= 128 else ("fma",),
                bwd_w="mma" if nin + 1 <= 128 and nout <= 128 else "fma",
                mma=(mma_grid, mma_grid * 8 * 16, 8 * 16), mma_need=-(-units // 8),
                splits=splits, rows_per_split=-(-rows // splits), split_need=-(-rows // 128))


def rad_route(edges, src, sms):
    """Radial forward (lgae_layers.cu:602: CTAs of LGAE_RAD_EB edges, at most 8 per SM) and adjoint (rad_ctas :544: at most
    LGAE_RAD_CTAS per SM, one partial row each)."""
    eb = src["rad_eb"]
    need = -(-edges // eb)
    fwd = max(1, min(need, 8 * sms))
    bwd = max(1, min(need, src["rad_ctas"] * sms))
    return dict(need=need, fwd=(fwd, fwd * eb, eb), bwd=(bwd, bwd * eb, eb))


def past_cap(work, grid_pass):
    """work exceeds one pass of the capped grid, and the last pass ends inside a CTA."""
    _, stride, per_cta = grid_pass
    return work > stride and (work % stride) % per_cta != 0


# ---------------------------------------------------------------------------------------------------------------------
# case tables (functions of the SM count)
# ---------------------------------------------------------------------------------------------------------------------
def _node(C, keys=IRREPS3):
    return {k: C for k in keys}


def cg_cases(sms):
    """Each case: node and edge irreps {key: channels}, batch (B, N) (point-wise: (rows,)), aggregate, swap (the edge operand
    first), maxdim.  The comment says what the case is there for; the table test checks the union."""
    E01, E0, E1, E014 = {(0, 0): 0, (1, 1): 0}, {(0, 0): 0}, {(1, 1): 0}, {(0, 0): 0, (1, 1): 0, (2, 2): 0}

    def ch(edge, C):
        return {k: C for k in edge}
    cases = {
        # point-wise past the grid cap: rows * C * 16 components (forward) and rows * C * 8 (adjoint) > 8 SMs x 256 threads
        "pt_cap": dict(node={(1, 1): 4}, edge={(1, 1): 4}, batch=(64 * sms + 5,), agg=False, swap=False, maxdim=3),
        # max_zf = 2 edges (D2T = 1 + 4 + 9): per-pair Kronecker kernels d2 = 1, 4, 9, edge adjoints, node adjoints (d1, 1|4)
        "zf2": dict(node=_node(3), edge=ch(E014, 3), batch=(2, 7), agg=True, swap=False, maxdim=3),
        "zf2_swap": dict(node=_node(3), edge=ch(E014, 3), batch=(2, 7), agg=True, swap=True, maxdim=3),
        # edge parts of d = 2 and 6 (CGDict(maxdim=3) has (1,0) and (2,1)): block kernels; d = 3 alone: Kronecker d2 = 3
        "edge_d2": dict(node={(0, 0): 2, (1, 1): 2, (1, 0): 2, (2, 1): 2}, edge={(1, 0): 2}, batch=(2, 6), agg=True, swap=False, maxdim=3),
        "edge_d6": dict(node={(0, 0): 2, (1, 1): 2, (2, 2): 2}, edge={(2, 1): 2}, batch=(2, 5), agg=True, swap=True, maxdim=3),
        "edge_d3": dict(node={(0, 0): 2, (2, 0): 2, (2, 2): 2}, edge={(2, 0): 2}, batch=(3, 5), agg=True, swap=False, maxdim=3),
        # mixed channel counts: (2,2) meets no partner below maxdim 2, so the call cannot take the one-launch kernel
        "mixed_channels": dict(node={(0, 0): 4, (1, 1): 4, (2, 2): 7}, edge=ch(E01, 4), batch=(2, 6), agg=True, swap=False, maxdim=2),
        # the jet slab is over 100 KB: neighbour-split forward, tiled adjoint.  Three jets, so that the grid's split of the
        # particles (ceil(2 SMs / B)) is smaller than N and does not divide it; "split" also needs more than one neighbour tile
        "split": dict(node={(2, 2): 4, (1, 1): 4}, edge={(1, 0): 4}, batch=(3, _split_n(240, 3, sms)), agg=True, swap=False, maxdim=3),
        "split_swap": dict(node={(2, 2): 4}, edge={(1, 0): 4}, batch=(3, _split_n(160, 3, sms)), agg=True, swap=True, maxdim=3),
        # the Kronecker kernels' K / gK buffers would exceed the shared memory of a CTA: block kernel / generic edge adjoint.
        # (1,1) x (2,2) at 245 channels: the forward's slab fits 100 KB, K does not fit next to it; (2,2) x (2,2) at 16 channels
        # (a max_zf = 2 model's pair): the edge adjoint's gK does not fit
        "kron_smem_fwd": dict(node={(1, 1): 245}, edge={(2, 2): 245}, batch=(2, 2), agg=True, swap=False, maxdim=3),
        "kron_smem_edge": dict(node={(2, 2): 16}, edge={(2, 2): 16}, batch=(2, 20), agg=True, swap=False, maxdim=3),
        # one-launch kernels: D2T = 1, 4, 5 (5 also from (1,0) + (2,0)); node adjoint D1T = 5 and 20
        "multi_d1": dict(node=_node(3), edge=ch(E0, 3), batch=(2, 9), agg=True, swap=False, maxdim=3),
        "multi_d4": dict(node=_node(3), edge=ch(E1, 3), batch=(2, 9), agg=True, swap=True, maxdim=3),
        "multi_d5_n5": dict(node=_node(4, [(0, 0), (1, 1)]), edge=ch(E01, 4), batch=(3, 11), agg=True, swap=False, maxdim=2),
        "multi_d5_odd_parts": dict(node=_node(2, [(0, 0), (1, 1), (1, 0), (2, 1)]), edge={(1, 0): 2, (2, 0): 2}, batch=(2, 6), agg=True,
                                   swap=False, maxdim=3),
        # N * C = 256 and 257 at D1T = 20: the node adjoint in one launch, then per pair
        "nc256": dict(node=_node(2), edge=ch(E01, 2), batch=(1, 128), agg=True, swap=False, maxdim=3),
        "nc257": dict(node=_node(1), edge=ch(E01, 1), batch=(1, 257), agg=True, swap=True, maxdim=3),
        # 16 channels: the ib loops of the one-launch kernels shrink their row blocks
        "multi_ib_shrink": dict(node=_node(16), edge=ch(E01, 16), batch=(2, 16), agg=True, swap=False, maxdim=3),
        # the one-launch forward needs more than 160 KB: LGAE_E_UNSUPPORTED, the pairs one by one (same numbers)
        "multi_fwd_fallback": dict(node=_node(16), edge=ch(E01, 16), batch=(1, 128), agg=True, swap=False, maxdim=3),
        # the forward fits, the one-launch adjoint does not: every gradient from the per-pair adjoint
        "multi_bwd_fallback": dict(node=_node(72), edge=ch(E01, 72), batch=(2, 2), agg=True, swap=True, maxdim=3),
    }
    return cases


def _split_n(n, B, sms):
    """The smallest N >= n that the neighbour-split forward's grid (split = ceil(2 SMs / B) CTAs over the particles) covers in
    more than one pass, the last one partial."""
    split = -(-2 * sms // B)
    return _first(n, lambda m: m > split and m % split != 0)


def _first(n, ok):
    """The smallest size >= n with ok(size): shapes derived from the SM count that also end their last pass mid-CTA."""
    while not ok(n):
        n += 1
    return n


def _mix_ragged(rows, cin, d, sms):
    def ok(r):
        m = mix_route(r, cin, 1, d, sms)
        return r % m["rows_per_cta"] != 0 and (r * d <= 8 * sms * 256 or (past_cap(r * d, m["fwd"]) and past_cap(r * cin * d, m["bwd_x"])))
    return _first(rows, ok)


def mix_cases(sms):
    """(rows, c_in, c_out, d); the weight gradient's CTAs (at most 4 per SM) take several rows each, the last one fewer."""
    return {
        # forward and bwd_x past the grid cap; COV 16 in two blocks of output channels (co0 = 0, 16)
        "cov16_cap": (_mix_ragged((8 * sms * 256) // 9 + 1, 3, 9, sms), 3, 20, 9),
        # COV 4, co_blk 4
        "cov4": (_mix_ragged(8 * sms + 1, 5, 4, sms), 5, 3, 4),
        # COV 8, co_blk 8
        "cov8": (_mix_ragged(12 * sms - 1, 6, 1, sms), 6, 7, 1),
        # COV 16 with one block (9 <= c_out <= 16), co_blk 8 over two passes
        "cov16_one_block": (_mix_ragged(4 * sms + 3, 12, 3, sms), 12, 12, 3),
    }


def sv_cases(sms):
    """(edges, cs, cv, d): past the grid cap of the forward (edges * C * d) and the adjoint (edges * (cs + cv * d))."""
    def case(cs, cv, d):
        works = (max(cs, cv) * d, cs + cv * d)
        e = _first((8 * sms * 256) // min(works) + 1, lambda e: all(past_cap(e * w, grid_stride_pass(e * w, 256, sms)) for w in works))
        return (e, cs, cv, d)
    return {"bcast_v": case(3, 1, 4), "same": case(3, 3, 4), "bcast_s": case(1, 3, 4)}


def lin_cases(sms):
    """(rows, n_in, n_out, slope)."""
    cap = 2 * 128 * sms + 77
    return {
        # MMA forward / bwd_x / bwd_w past their caps (grid and lin_splits); NT 4 and 12
        "mma_cap": (cap, 30, 96, 0.01),
        # FMA bwd_w (n_in + 1 > 128) past lin_splits, MMA forward NT 2 / bwd_x NT 16
        "fma_w_cap": (cap, 128, 12, None),
        # FMA forward and bwd_x (n_out > 128): the widths of a 12-channel MLP (2C' = 24 -> 6 x 24 = 144)
        "fma_144": (700, 24, 144, 0.01),
        "fma_144_back": (701, 144, 24, None),
        # tile widths NT 8 (forward) / NT 4 (bwd_x), one short row group
        "nt8": (37, 27, 60, 0.2),
    }


def rad_cases(sms):
    """(basis, max_zf, num_basis_fn, C, B, N): edges = B N N (Cartesian) or 2 B N N (canonical), past 8 SMs x 64 edges."""
    def b_for(n, per):
        return -(-(8 * sms * 64) // (per * n * n)) + 1
    return {
        "cartesian_cap": ("cartesian", 1, 10, 4, b_for(30, 1), 30),
        # 20 basis functions (k2 = 40 > 32), three zonal degrees
        "canonical_k40_cap": ("canonical", 2, 20, 3, b_for(29, 2), 29),
    }


MODEL_CASES = {
    # max_zf = 2 (edges (0,0) + (1,1) + (2,2)): the per-pair aggregated kernels inside the model, three radial outputs.  Encoder
    # only: the decoder's input zonal functions then include (2,2), which its input mix has no weight for, and the oracle (as the
    # reference's MixReps) refuses that rep, so the decoder keeps max_zf = 1
    "maxdim3_zf2": dict(seed=71, batch=2, n=6, maxdim=3, max_zf=2, dec_max_zf=1, num_basis_fn=3, enc_channels=[2, 3, 2], dec_channels=[2, 2, 3],
                        tau_s=1, tau_v=2, map_to_latent="mean", mlp_depth=1, mlp_width=2),
    # 12 channels: mix COV 16, MLP widths 6 x 24 = 144 (plain-FMA linear kernels)
    "channels12": dict(seed=72, batch=3, n=7, maxdim=2, max_zf=1, num_basis_fn=3, enc_channels=[12, 9, 4], dec_channels=[4, 16, 10],
                       tau_s=2, tau_v=3, map_to_latent="min&max", mlp_depth=1, mlp_width=6),
    # 20 radial basis functions (k2 = 40 > 32)
    "basis20": dict(seed=73, batch=2, n=8, maxdim=2, max_zf=1, num_basis_fn=20, enc_channels=[3, 4, 3], dec_channels=[3, 4, 2],
                    tau_s=1, tau_v=2, map_to_latent="max", mlp_depth=1, mlp_width=2),
}

CFG4 = dict(B=1024, N=30, enc=[6, 6, 8, 8], dec=[8, 8, 6, 6], num_basis_fn=10, mlp_depth=6, mlp_width=6)


def cfg4_check_jets(sms):
    """The jets of the cfg-4 step whose rows the last grid-stride pass of the capped launchers reads, with the first and
    the last jet: the point-wise CG square of (1,1) x (1,1) at 8 channels (node rows, 16 components each), scalar x irrep at 8
    channels and d = 4 (edges), the radial forward and adjoint (edges)."""
    B, N = CFG4["B"], CFG4["N"]
    rows, edges = B * N, B * N * N
    jets = {0, B - 1}
    for work, per_row, grid_pass, per_jet in (
            (rows * 8 * 16, 8 * 16, grid_stride_pass(rows * 8 * 16, 256, sms), N),       # cg_pt_fwd, (1,1) x (1,1), C = 8
            (edges * 8 * 4, 8 * 4, grid_stride_pass(edges * 8 * 4, 256, sms), N * N),     # sv_fwd, C = 8, d = 4
            (edges, 1, (8 * sms, 8 * sms * 64, 64), N * N),                               # radial forward
            (edges, 1, (4 * sms, 4 * sms * 64, 64), N * N)):                              # radial adjoint
        last = ((work - 1) // grid_pass[1]) * grid_pass[1]
        jets.add(last // per_row // per_jet)
        jets.add(min(B - 1, last // per_row // per_jet + 1))
    k = 1
    while len(jets) < 8:   # fill up with jets spread over the batch
        jets.add((k * 131) % B)
        k += 1
    return sorted(jets)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the tables reach every branch
# ---------------------------------------------------------------------------------------------------------------------
_CG = None


def _cgdict():
    global _CG
    if _CG is None:
        from lgn_autoencoder_b200.cg_lib import CGDict
        _CG = CGDict(maxdim=3, transpose=True, dtype=torch.float64, device=torch.device("cpu"))
    return _CG


def test_case_tables_reach_every_branch():
    sms = B200_SMS
    src = source_instances()
    assert src["kron_fwd"] and src["kron_edge"] and src["kron_node"] and src["multi_fwd"] and src["lin"]
    # --- CG product: every instance and branch of the per-pair, one-launch and fallback paths
    seen, smem = set(), []
    for name, case in cg_cases(sms).items():
        for what, kernel, nbytes, info in cg_route(case, src, sms):
            smem.append((nbytes, name, kernel))
            seen.add((what, kernel))
            if what == "multi":
                seen.add(("ib", kernel, info))
            elif what == "node_ok":
                seen.add(("node_ok", kernel) + info)
            elif what == "fwd" and info == "kron_too_big":
                seen.add(("fwd", "kron_too_big"))
            elif what == "fwd" and kernel == "split":
                # past the cap of its grid (several particles per CTA, the last pass partial), more than one neighbour tile
                seen.add(("split_past_cap", info["n"] > info["split"] and info["n"] % info["split"] != 0))
                seen.add(("split_tiles", info["jt"] < info["n"]))
            elif what == "pt_work":
                seen.add(("pt_past_cap", kernel, past_cap(info, grid_stride_pass(info, 256, sms))))
    want = {("fwd", k) for k in ["pointwise", "block", "split", "kron_too_big"] + [f"kron{d}" for d in src["kron_fwd"]]}
    want |= {("bwd", k) for k in ["pointwise", "edge_generic", "edge_generic_kron_too_big", "tiled"] + [f"edge_kron{d}" for d in src["kron_edge"]]}
    want |= {("bwd", ("node_kron", a, b)) for a, b in src["kron_node"]}
    want |= {("multi", f"multi_fwd{d}") for d in src["multi_fwd"]} | {("multi", f"multi_edge{d}") for d in src["multi_edge"]}
    want |= {("multi", f"multi_node{a}") for a, _ in src["multi_node"]}
    want |= {("fallback", "fwd"), ("fallback", "bwd"), ("split_past_cap", True), ("split_tiles", True)}
    want |= {("pt_past_cap", "fwd", True), ("pt_past_cap", "bwd", True)}
    assert want <= seen, sorted(map(str, want - seen))
    # every launch fits the shared memory of a CTA
    assert max(smem)[0] <= SMEM_MAX, max(smem)
    # N * C = 256 and 257 at D1T = 20 on both sides of node_ok
    assert ("node_ok", True, 20, 256) in seen and ("node_ok", False, 20, 257) in seen
    # the ib loops shrink below their starting value (forward, edge and node adjoints)
    ibs = [k for k in seen if k[0] == "ib"]
    assert any(k[1].startswith("multi_fwd") and k[2] < src["agg_fwd_ib"] for k in ibs)
    assert any(k[1].startswith("multi_edge") and k[2] < src["agg_edge_ib"] for k in ibs)
    assert any(k[1].startswith("multi_node") and k[2] < 2 for k in ibs)
    # --- mix: COV 4/8/16, co_blk 4/8, several output blocks, rows_per_cta > 1 with a short last CTA, grid caps
    mr = {name: mix_route(*c, sms) for name, c in mix_cases(sms).items()}
    assert {r["cov"] for r in mr.values()} == {4, 8, 16} and {r["co_blk"] for r in mr.values()} == {4, 8}
    assert any(r["co_blocks"] > 1 for r in mr.values())
    for name, (rows, cin, cout, d) in mix_cases(sms).items():
        r = mr[name]
        assert rows > 4 * sms and r["rows_per_cta"] > 1 and rows % r["rows_per_cta"] != 0, name
    rows, cin, cout, d = mix_cases(sms)["cov16_cap"]
    assert past_cap(rows * d, mr["cov16_cap"]["fwd"]) and past_cap(rows * cin * d, mr["cov16_cap"]["bwd_x"])
    # --- scalar x irrep past the cap, all three broadcasts
    for e, cs, cv, d in sv_cases(sms).values():
        C = max(cs, cv)
        assert past_cap(e * C * d, grid_stride_pass(e * C * d, 256, sms)) and past_cap(e * (cs + cv * d), grid_stride_pass(e * (cs + cv * d), 256, sms))
    assert {(cs == 1, cv == 1) for _, cs, cv, _ in sv_cases(sms).values()} == {(False, True), (False, False), (True, False)}
    # --- linear: MMA / FMA for forward, bwd_x and bwd_w, every LGAE_LIN tile width, caps of the MMA grid and lin_splits
    lr = {name: lin_route(r, i, o, sms, src["lin"]) for name, (r, i, o, _) in lin_cases(sms).items()}
    nts = {r["fwd"][1] for r in lr.values() if r["fwd"][0] == "mma"} | {r["bwd_x"][1] for r in lr.values() if r["bwd_x"][0] == "mma"}
    assert nts == src["lin"], src["lin"] - nts
    assert {r["fwd"][0] for r in lr.values()} == {r["bwd_x"][0] for r in lr.values()} == {"mma", "fma"}
    assert {r["bwd_w"] for r in lr.values()} == {"mma", "fma"}
    capped = [n for n, r in lr.items() if r["split_need"] > sms and lin_cases(sms)[n][0] % r["rows_per_split"] != 0]
    assert {lr[n]["bwd_w"] for n in capped} == {"mma", "fma"}, capped
    assert any(r["mma_need"] > sms and past_cap(-(-lin_cases(sms)[n][0] // 16) * 16, r["mma"]) for n, r in lr.items() if r["fwd"][0] == "mma")
    # --- radial functions past the caps of the forward and the adjoint, k2 > 32
    for basis, zf, nb, C, B, N in rad_cases(sms).values():
        e = B * N * N * (2 if basis == "canonical" else 1)
        r = rad_route(e, src, sms)
        assert past_cap(e, r["fwd"]) and past_cap(e, r["bwd"]), (basis, e)
    assert {c[0] for c in rad_cases(sms).values()} == {"cartesian", "canonical"} and max(2 * c[2] for c in rad_cases(sms).values()) > 32
    # --- composite-only models: max_zf 2, 9-16 channels, 17-20 radial basis functions (none of them fused)
    assert any(c["max_zf"] == 2 and c["maxdim"] == 3 for c in MODEL_CASES.values())
    assert any(9 <= max(c["enc_channels"] + c["dec_channels"]) <= 16 for c in MODEL_CASES.values())
    assert any(17 <= c["num_basis_fn"] <= 20 for c in MODEL_CASES.values())
    assert any(2 * c["mlp_width"] * max(c["enc_channels"][1:] + c["dec_channels"][1:]) > 128 for c in MODEL_CASES.values())
    # --- the cfg-4 step's jets for the oracle: first, last and the last grid-stride passes
    jets = cfg4_check_jets(sms)
    assert 0 in jets and CFG4["B"] - 1 in jets and len(jets) <= 10


def test_kronecker_launches_fit_shared_memory():
    """No GPU: for every (node irrep, edge irrep) pair of CGDict(maxdim=3), every channel count the host code accepts and every
    jet size that takes a whole-jet forward or the one-launch edge adjoint, the launch the rules above pick fits the shared
    memory of a CTA (the Kronecker kernels' K / gK buffers come on top of the 100 KB their choice is made on)."""
    from lgn_autoencoder_b200 import layer_ops
    src = source_instances()
    keys = [(k, n) for k in range(3) for n in range(3)]
    worst = (0, None)
    for node in keys:
        for edge in keys:
            outs = [(k, n) for k in range(abs(node[0] - edge[0]), min(3, node[0] + edge[0] + 1), 2)
                    for n in range(abs(node[1] - edge[1]), min(3, node[1] + edge[1] + 1), 2)]
            if not outs:
                continue
            terms, n_comp = layer_ops._pair_terms(_cgdict(), node, edge, outs, False)
            d1, d2 = _dim(node), _dim(edge)
            for C in range(1, 4 * 256 // max(n_comp, d1) + 1):
                for nj in range(1, 100 * KB // (16 * C * d1) + 2):
                    launches = []
                    if terms_doubles(len(terms), n_comp + 1) * 8 + nj * C * (d1 + d2) * 16 <= 100 * KB:
                        launches.append(cg_pair_fwd(C, d1, d2, n_comp, len(terms), 1, nj, src["kron_fwd"], B200_SMS)[:2])
                    if terms_doubles(len(terms), d2 + 1) * 8 + (nj * C * d1 + min(8, nj) * C * n_comp) * 16 <= 100 * KB:
                        launches += cg_pair_bwd(C, d1, d2, n_comp, len(terms), nj, False, True, src["kron_edge"], src["kron_node"])
                    for name, nbytes in launches:
                        worst = max(worst, (nbytes, (node, edge, C, nj, name)))
    assert worst[0] <= SMEM_MAX, worst


def test_cg_reference_matches_oracle():
    """No GPU: the einsum restatement below (used for the shapes the oracle's materialised Kronecker product cannot take) gives
    the oracle's cg_product and its gradients on small shapes, both orientations and point-wise."""
    from oracle import lgae_oracle as orc
    gen = torch.Generator().manual_seed(3)
    node = _rand_rep(gen, (2, 5), {(0, 0): 2, (1, 1): 2, (2, 2): 2, (1, 0): 2})
    edge = _rand_rep(gen, (2, 5, 5), {(0, 0): 2, (1, 1): 2, (2, 1): 2})
    cgt = orc.cg_table(3)
    for a, b, agg in ((node, edge, True), (edge, node, True), (node, node, False)):
        ref = orc.cg_product(cgt, a, b, 3, agg)
        mine = ref_cg_product(cgt, a, b, 3, agg)
        assert list(mine) == list(ref)
        scale = max(v.abs().max().item() for v in ref.values())   # the square has parts that vanish exactly: rounding level only
        for k in ref:
            assert (mine[k] - ref[k]).abs().max().item() < 1e-13 * scale, k
        cot = {k: torch.randn(v.shape, generator=gen, dtype=torch.float64) for k, v in ref.items()}
        leaves = list(a.values()) + ([] if b is a else list(b.values()))
        g1 = torch.autograd.grad(sum((ref[k] * cot[k]).sum() for k in ref), leaves, allow_unused=True)
        g2 = torch.autograd.grad(sum((mine[k] * cot[k]).sum() for k in mine), leaves, allow_unused=True)
        for x, y in zip(g1, g2):
            assert (x is None) == (y is None) and (x is None or rel_err(y, x) < 1e-13)


# ---------------------------------------------------------------------------------------------------------------------
# references and helpers
# ---------------------------------------------------------------------------------------------------------------------
def _rand_rep(gen, batch, tau, requires_grad=True):
    return {k: torch.randn((2,) + batch + (c, _dim(k)), generator=gen, dtype=torch.float64).requires_grad_(requires_grad) for k, c in tau.items()}


def _cmul_einsum(eq, x, y):
    return torch.stack([torch.einsum(eq, x[0], y[0]) - torch.einsum(eq, x[1], y[1]), torch.einsum(eq, x[0], y[1]) + torch.einsum(eq, x[1], y[0])])


def ref_cg_product(cgt, rep1, rep2, maxdim, aggregate):
    """cg_ops.py:135-218 as the oracle states it, with the neighbour sum taken before the CG matrix (an einsum instead of the
    materialised Kronecker product): out[(k,n)] = H . sum_j z1 (x) z2, pairs in loop order, channel-concatenated."""
    maxk1, maxn1 = max(k for k, _ in rep1), max(n for _, n in rep1)
    maxk2, maxn2 = max(k for k, _ in rep2), max(n for _, n in rep2)
    max_dim = min(max(maxk1 + maxk2, maxn1 + maxn2) + 1, maxdim)
    out = {}
    for (k1, n1), z1 in rep1.items():
        for (k2, n2), z2 in rep2.items():
            if max(k1, n1, k2, n2) > max_dim - 1:
                continue
            keys = [(k, n) for k in range(abs(k1 - k2), min(maxdim, k1 + k2 + 1), 2) for n in range(abs(n1 - n2), min(maxdim, n1 + n2 + 1), 2)]
            if not keys:
                continue
            h = torch.cat([cgt[((k1, n1), (k2, n2))][key] for key in keys], -2)
            if not aggregate:
                kr = _cmul_einsum("...ca,...cd->...cad", z1, z2)
            elif z1.dim() == z2.dim() + 1:
                kr = _cmul_einsum("bijca,bjcd->bicad", z1, z2)
            else:
                kr = _cmul_einsum("bjca,bijcd->bicad", z1, z2)
            kr = kr.reshape(kr.shape[:-2] + (-1,))
            dec = torch.einsum("mk,...k->...m", h, kr)
            for key, piece in zip(keys, torch.split(dec, [_dim(k) for k in keys], dim=-1)):
                out.setdefault(key, []).append(piece)
    return {key: torch.cat(v, dim=-2) for key, v in out.items()}


def _assert_sum_close(got, ref, absref, n, what):
    """Element-wise a-priori bound of two recursive fp64 sums of n terms: |got - ref| <= 2 n u sum|term| (+ a denormal floor)."""
    err = (got.detach().cpu() - ref.detach()).abs()
    bound = 2 * n * U * absref.detach() + 1e-300
    worst = (err / bound).max().item()
    assert worst <= 1.0, (what, worst, err.max().item())


def _dev():
    return torch.device("cuda:0")


def _sms():
    from lgn_autoencoder_b200 import _lib
    return int(_lib.load().lgae_device_sm_count())


def _to_dev(rep):
    return {k: v.detach().to(_dev()).requires_grad_(True) for k, v in rep.items()}


# ---------------------------------------------------------------------------------------------------------------------
# GPU: layer ops against fp64 references
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(cg_cases(B200_SMS)))
def test_cg_product_cases_match_reference(name):
    """cg_product (public API -> layer_ops._CGPairsFn) against ref_cg_product on the CPU: every output part and the gradient of
    every operand part; the adjoint again, bit-identical (fixed summation order)."""
    from lgn_autoencoder_b200.cg_lib import cg_product
    from lgn_autoencoder_b200.g_lib import GVec
    from oracle import lgae_oracle as orc
    case = cg_cases(_sms())[name]
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    if case["agg"]:
        B, N = case["batch"]
        node = _rand_rep(gen, (B, N), case["node"])
        edge = _rand_rep(gen, (B, N, N), case["edge"])
    else:
        node = _rand_rep(gen, case["batch"], case["node"])
        edge = _rand_rep(gen, case["batch"], case["edge"])
    rep1, rep2 = (edge, node) if case["swap"] else (node, edge)
    maxdim = case["maxdim"]
    ref = ref_cg_product(orc.cg_table(3), rep1, rep2, maxdim, case["agg"])
    cot = {k: torch.randn(v.shape, generator=gen, dtype=torch.float64) for k, v in ref.items()}
    leaves = list(rep1.values()) + list(rep2.values())
    g_ref = torch.autograd.grad(sum((ref[k] * cot[k]).sum() for k in ref), leaves, allow_unused=True)

    d1, d2 = _to_dev(rep1), _to_dev(rep2)
    cg = _cgdict().to(device=_dev())

    def run():
        out = cg_product(cg, GVec(d1, ignore_check=True), GVec(d2, ignore_check=True), maxdim=maxdim, aggregate=case["agg"])
        g = torch.autograd.grad(sum((out[k] * cot[k].to(_dev())).sum() for k in out.keys()), list(d1.values()) + list(d2.values()),
                                allow_unused=True)
        return out, g
    out, g = run()
    assert list(out.keys()) == list(ref.keys())
    for k in ref:
        assert rel_err(out[k], ref[k]) < TOL, (name, k)
    for i, (a, b) in enumerate(zip(g, g_ref)):
        if b is None:
            assert a is None or a.abs().max().item() == 0.0, (name, i)
        else:
            assert rel_err(a, b) < TOL, (name, i)
    out2, g2 = run()
    for k in ref:
        assert torch.equal(out[k], out2[k]), (name, k)
    for a, b in zip(g, g2):
        assert (a is None and b is None) or torch.equal(a, b), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(mix_cases(B200_SMS)))
def test_mix_cases_match_reference(name):
    """layer_ops.mix against the oracle's mix_zweight_zvec: output and dx within 1e-12 (sums of c_out / c_in products); dW, a sum
    over rows * d terms, within the bound of that sum length, and bit-identical when repeated."""
    from lgn_autoencoder_b200 import layer_ops
    from oracle import lgae_oracle as orc
    rows, cin, cout, d = mix_cases(_sms())[name]
    gen = torch.Generator().manual_seed(rows)
    w = torch.randn((2, cout, cin), generator=gen, dtype=torch.float64, requires_grad=True)
    x = torch.randn((2, rows, cin, d), generator=gen, dtype=torch.float64, requires_grad=True)
    ref = orc.mix_zweight_zvec(w, x)
    cot = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    gw_ref, gx_ref = torch.autograd.grad((ref * cot).sum(), (w, x))
    # sum of |terms| of dW[co, ci] = sum_{r,m} conj(x) g: |x| |g| summed (re and im parts alike)
    ax, ag = x.detach().abs().sum(0), cot.abs().sum(0)
    gw_abs = torch.einsum("rcm,rom->oc", ax, ag).expand(2, cout, cin)
    wd, xd = w.detach().to(_dev()).requires_grad_(True), x.detach().to(_dev()).requires_grad_(True)
    out = layer_ops.mix(wd, xd)
    gw, gx = torch.autograd.grad((out * cot.to(_dev())).sum(), (wd, xd))
    assert rel_err(out, ref) < TOL and rel_err(gx, gx_ref) < TOL, name
    _assert_sum_close(gw, gw_ref, gw_abs, 2 * rows * d, name)
    gw2, gx2 = torch.autograd.grad((layer_ops.mix(wd, xd) * cot.to(_dev())).sum(), (wd, xd))
    assert torch.equal(gw, gw2) and torch.equal(gx, gx2), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(sv_cases(B200_SMS)))
def test_scalar_irrep_cases_match_reference(name):
    """layer_ops.scalar_irrep past its grid cap against the oracle's mul_zscalar_zirrep (broadcast sums: at most C * d terms)."""
    from lgn_autoencoder_b200 import layer_ops
    from oracle import lgae_oracle as orc
    e, cs, cv, d = sv_cases(_sms())[name]
    gen = torch.Generator().manual_seed(e + cs)
    s = torch.randn((2, e, cs), generator=gen, dtype=torch.float64, requires_grad=True)
    v = torch.randn((2, e, cv, d), generator=gen, dtype=torch.float64, requires_grad=True)
    ref = orc.mul_zscalar_zirrep(s, v)
    cot = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    gs_ref, gv_ref = torch.autograd.grad((ref * cot).sum(), (s, v))
    sd, vd = s.detach().to(_dev()).requires_grad_(True), v.detach().to(_dev()).requires_grad_(True)
    out = layer_ops.scalar_irrep(sd, vd)
    gs, gv = torch.autograd.grad((out * cot.to(_dev())).sum(), (sd, vd))
    assert rel_err(out, ref) < TOL and rel_err(gs, gs_ref) < TOL and rel_err(gv, gv_ref) < TOL, name
    gs2, gv2 = torch.autograd.grad((layer_ops.scalar_irrep(sd, vd) * cot.to(_dev())).sum(), (sd, vd))
    assert torch.equal(gs, gs2) and torch.equal(gv, gv2), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(lin_cases(B200_SMS)))
def test_linear_cases_match_torch_fp64(name):
    """layer_ops.linear against torch fp64 on the CPU: y and dx within 1e-12 (sums of n_in / n_out products); dW and db, sums
    over all rows, within the bound of that sum length and bit-identical when repeated."""
    from lgn_autoencoder_b200 import layer_ops
    rows, nin, nout, slope = lin_cases(_sms())[name]
    gen = torch.Generator().manual_seed(rows + nin)
    x = torch.randn((rows, nin), generator=gen, dtype=torch.float64, requires_grad=True)
    w = torch.randn((nout, nin), generator=gen, dtype=torch.float64, requires_grad=True)
    b = torch.randn((nout,), generator=gen, dtype=torch.float64, requires_grad=True)
    ref = torch.nn.functional.linear(x, w, b)
    if slope is not None:
        ref = torch.nn.functional.leaky_relu(ref, slope)
    cot = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    gx_ref, gw_ref, gb_ref = torch.autograd.grad((ref * cot).sum(), (x, w, b))
    dz = cot if slope is None else torch.where(ref > 0, cot, cot * slope)
    gw_abs, gb_abs = dz.abs().t() @ x.detach().abs(), dz.abs().sum(0)
    xd, wd, bd = (t.detach().to(_dev()).requires_grad_(True) for t in (x, w, b))
    out = layer_ops.linear(xd, wd, bd, leaky_slope=slope)
    gx, gw, gb = torch.autograd.grad((out * cot.to(_dev())).sum(), (xd, wd, bd))
    assert rel_err(out, ref) < TOL and rel_err(gx, gx_ref) < TOL, name
    _assert_sum_close(gw, gw_ref, gw_abs, rows, name + "/dW")
    _assert_sum_close(gb, gb_ref, gb_abs, rows, name + "/db")
    gx2, gw2, gb2 = torch.autograd.grad((layer_ops.linear(xd, wd, bd, leaky_slope=slope) * cot.to(_dev())).sum(), (xd, wd, bd))
    assert torch.equal(gx, gx2) and torch.equal(gw, gw2) and torch.equal(gb, gb2), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(rad_cases(B200_SMS)))
def test_radial_cases_match_oracle(name):
    """RadPolyTrig past the caps of the radial forward and adjoint against the oracle's rad_poly_trig: outputs within 1e-12
    (sums of k2 products), d/dnorms within 1e-12, the parameter gradients (sums over all edges) within the bound of that sum
    length and bit-identical when repeated."""
    from lgn_autoencoder_b200.nn import RadPolyTrig
    from oracle import lgae_oracle as orc
    basis, zf, nb, C, B, N = rad_cases(_sms())[name]
    gen = torch.Generator().manual_seed(B * N)
    torch.manual_seed(nb)
    mod = RadPolyTrig(zf, nb, C, mix=True, input_basis=basis, device=_dev(), dtype=torch.float64)
    shape = (B, N, N) if basis == "cartesian" else (2, B, N, N)
    norms = torch.randn(shape, generator=gen, dtype=torch.float64)
    mask = (torch.rand((B, N, N), generator=gen) > 0.3).to(torch.uint8)
    params = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in mod.named_parameters()}
    names = list(params)
    x_ref = norms.clone().requires_grad_(True)
    lin = [(params[f"linear.{l}.weight"], params[f"linear.{l}.bias"]) for l in range(zf + 1)]
    ref = orc.rad_poly_trig(x_ref, mask, params["a"], params["b"], params["c"], lin, C, basis)
    cot = {k: torch.randn(v.shape, generator=gen, dtype=torch.float64) for k, v in ref.items()}
    g_ref = torch.autograd.grad(sum((ref[k] * cot[k]).sum() for k in ref), [x_ref] + [params[n] for n in names])
    # sum of |terms| of every parameter gradient: the same contraction on absolute values
    abs_params = {n: p.detach().abs() for n, p in params.items()}
    abs_lin = [(abs_params[f"linear.{l}.weight"], abs_params[f"linear.{l}.bias"]) for l in range(zf + 1)]
    x_abs = norms.clone().requires_grad_(True)
    p_abs = {n: abs_params[n].clone().requires_grad_(True) for n in names}
    bells_abs = _rad_abs_terms(x_abs, mask, p_abs, abs_lin, zf, C, basis, cot)

    x = norms.to(_dev()).requires_grad_(True)
    mparams = dict(mod.named_parameters())

    def run():
        out = mod(x, mask.to(_dev()))
        return out, torch.autograd.grad(sum((out[k] * cot[k].to(_dev())).sum() for k in ref), [x] + [mparams[n] for n in names])
    out, g = run()
    for k in ref:
        assert out[k].shape == ref[k].shape and rel_err(out[k], ref[k]) < TOL, (name, k)
    assert rel_err(g[0], g_ref[0]) < TOL, name
    edges = norms.numel()
    for n, a, r in zip(names, g[1:], g_ref[1:]):
        _assert_sum_close(a, r, bells_abs[n], edges * ((zf + 1) * (2 * C if basis == "cartesian" else C) + 1), (name, n))
    _, g2 = run()
    for a, b in zip(g, g2):
        assert torch.equal(a, b), name


def _rad_abs_terms(x, mask, p_abs, abs_lin, zf, C, basis, cot):
    """For every parameter, the sum over edges (and outputs) of the absolute values of the terms of its gradient: the
    derivative chain of rad_poly_trig with every factor replaced by its absolute value."""
    s = tuple(x.shape)
    m = mask.bool().unsqueeze(-1)
    xv = x.detach().unsqueeze(-1)
    a, b, c = p_abs["a"], p_abs["b"], p_abs["c"]
    r = (1 + (c.detach() * xv) ** 2 + 1e-16) ** -1
    bell = torch.where(m, b.detach() * r + a.detach(), torch.zeros(()))        # |bell| <= |b| r + |a|
    bell = bell.view(s + (1, -1))
    if basis == "canonical":
        g = [cot[(l, l)].abs() for l in range(zf + 1)]                           # (2,B,N,N,C)
    else:
        g = [cot[(l, l)].abs().permute(1, 2, 3, 4, 0).reshape(s + (2 * C,)) for l in range(zf + 1)]
    out = {}
    gb_abs = 0
    for l in range(zf + 1):
        gl = g[l].reshape(-1, g[l].shape[-1])
        bl = bell.reshape(-1, bell.shape[-1])
        out[f"linear.{l}.weight"] = gl.t() @ bl
        out[f"linear.{l}.bias"] = gl.sum(0)
        gb_abs = gb_abs + (g[l] @ abs_lin[l][0]).view(s + (1, -1))
    gb_abs = torch.where(m.unsqueeze(-2), gb_abs, torch.zeros(()))
    rr = r.view(s + (1, -1))
    xx = xv.view(s + (1, 1))
    out["a"] = gb_abs.reshape(-1, gb_abs.shape[-1]).sum(0).view(a.shape)
    out["b"] = (gb_abs * rr).reshape(-1, gb_abs.shape[-1]).sum(0).view(b.shape)
    out["c"] = (gb_abs * 2 * b.detach().view(1, -1) * rr * rr * c.detach().view(1, -1) * xx * xx).reshape(-1, gb_abs.shape[-1]).sum(0).view(c.shape)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# GPU: models only the composite trains
# ---------------------------------------------------------------------------------------------------------------------
def _build_model(cfg, dev):
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    torch.manual_seed(cfg["seed"])
    common = dict(maxdim=[cfg["maxdim"]], num_basis_fn=cfg["num_basis_fn"], weight_init="randn", level_gain=[1.0], activation="leakyrelu",
                  mlp=True, mlp_depth=cfg["mlp_depth"], mlp_width=cfg["mlp_width"], device=torch.device("cpu"), dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=cfg["n"], tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=cfg["tau_s"],
                     tau_latent_vectors=cfg["tau_v"], num_channels=cfg["enc_channels"], jet_features=False, map_to_latent=cfg["map_to_latent"],
                     max_zf=[cfg["max_zf"]], **common)
    mult = 2 if cfg["map_to_latent"] == "min&max" else 1
    dec = LGNDecoder(tau_latent_scalars=cfg["tau_s"] * mult, tau_latent_vectors=cfg["tau_v"] * mult, num_output_particles=cfg["n"],
                     tau_output_scalars=1, tau_output_vectors=1, num_channels=cfg["dec_channels"], cg_dict=enc.cg_dict,
                     max_zf=[cfg.get("dec_max_zf", cfg["max_zf"])], **common)
    return enc.to(dev), dec.to(dev)


def _oracle(enc, dec, cfg, p4, want_grads=True):
    """Oracle forward (and parameter gradients of the chamfer loss, 'sum' get_real) of one set of jets."""
    from oracle import lgae_oracle as orc
    enc_sd = {k: v.detach().cpu().clone().requires_grad_(want_grads) for k, v in enc.state_dict().items()}
    dec_sd = {k: v.detach().cpu().clone().requires_grad_(want_grads) for k, v in dec.state_dict().items()}
    ecfg = dict(num_channels=cfg["enc_channels"], maxdim=[cfg["maxdim"]], max_zf=[cfg["max_zf"]], map_to_latent=cfg["map_to_latent"])
    dcfg = dict(num_channels=cfg["dec_channels"], maxdim=[cfg["maxdim"]], max_zf=[cfg.get("dec_max_zf", cfg["max_zf"])])
    with torch.set_grad_enabled(want_grads):
        latent = orc.encoder_forward(enc_sd, ecfg, {"p4": p4})
        recon = orc.decoder_forward(dec_sd, dcfg, latent)
        loss = orc.chamfer_loss(orc.get_real(recon, "sum"), p4)
    grads = None
    if want_grads:
        loss.backward()
        grads = {"enc": {k: v.grad for k, v in enc_sd.items()}, "dec": {k: v.grad for k, v in dec_sd.items()}}
    return {k: v.detach() for k, v in latent.items()}, recon.detach(), loss.detach(), grads


def _param_grads(models):
    return {kind: {k: torch.zeros_like(p) if p.grad is None else p.grad.detach().clone() for k, p in m.named_parameters()}
            for kind, m in models.items()}


def _zero_grads(models):
    for m in models.values():
        for p in m.parameters():
            p.grad = None


@pytest.fixture(scope="module")
def cfg4_run():
    """cfg-4 exactly as bench.py extra_cfg4 builds it (seed 0, enc 6-6-8-8 / dec 8-8-6-6, 'mix', MLP 6 x 6, 10 basis functions,
    batch 1024 of its synthetic jets) through train.training_step."""
    from bench import synthetic_jets
    from lgn_autoencoder_b200.models import LGNDecoder, LGNEncoder
    from lgn_autoencoder_b200.train import training_step
    dev = _dev()
    B, N = CFG4["B"], CFG4["N"]
    torch.manual_seed(0)
    common = dict(maxdim=[3], num_basis_fn=CFG4["num_basis_fn"], max_zf=[1], weight_init="randn", level_gain=[1.0], activation="leakyrelu",
                  mlp=True, mlp_depth=CFG4["mlp_depth"], mlp_width=CFG4["mlp_width"], device=dev, dtype=torch.float64)
    enc = LGNEncoder(num_input_particles=N, tau_input_scalars=1, tau_input_vectors=1, tau_latent_scalars=1, tau_latent_vectors=8,
                     num_channels=CFG4["enc"], jet_features=False, map_to_latent="mix", **common)
    dec = LGNDecoder(tau_latent_scalars=1, tau_latent_vectors=8, num_output_particles=N, tau_output_scalars=1, tau_output_vectors=1,
                     num_channels=CFG4["dec"], cg_dict=enc.cg_dict, **common)
    assert not enc.fused and not dec.fused and enc.fused_forward and dec.fused_forward
    p4 = synthetic_jets(B, N, seed=2).to(dev)
    models = {"enc": enc, "dec": dec}
    _zero_grads(models)
    loss, recon, p4n = training_step(enc, dec, p4, l1_lambda=0.0, get_real="sum")
    jets = cfg4_check_jets(_sms())
    cfg = dict(enc_channels=CFG4["enc"], dec_channels=CFG4["dec"], maxdim=3, max_zf=1, map_to_latent="mix")
    return dict(enc=enc, dec=dec, models=models, p4=p4, p4n=p4n.detach(), loss=loss, recon=recon, jets=jets, cfg=cfg)


@pytest.mark.gpu
def test_cfg4_batch1024_forward_matches_fused_forward_and_oracle(cfg4_run):
    """Every jet: latents and reconstruction of the composite (the training call) against the fused maxdim-3 forward of the same
    model under no_grad (1e-10).  A few jets -- first, last, and those the last grid-stride pass of the capped launchers
    reads -- against the CPU oracle (1e-10)."""
    from lgn_autoencoder_b200 import fused
    r = cfg4_run
    enc, dec, p4n = r["enc"], r["dec"], r["p4n"]
    with torch.no_grad():
        lat_f = enc({"p4": p4n})
        recon_f = dec(lat_f)
    # the composite's latent of the same call
    lat_c = enc({"p4": p4n})
    recon = r["recon"].detach()
    for key in ((0, 0), (1, 1)):
        assert rel_err(lat_c[key], lat_f[key]) < 1e-10, key
    assert rel_err(recon, recon_f) < 1e-10
    # per jet as well: a wrong jet must not hide behind the max-norm of the whole batch
    per_jet = (recon - recon_f).abs().amax(dim=(0, 2, 3)) / recon_f.abs().amax(dim=(0, 2, 3))
    assert per_jet.max().item() < 1e-10, per_jet.argmax().item()
    assert abs(r["loss"].item() - fused.chamfer_loss(recon_f, p4n, "sum").item()) <= 1e-10 * abs(r["loss"].item())
    for j in r["jets"]:
        lat_o, recon_o, _, _ = _oracle(enc, dec, r["cfg"], p4n[j:j + 1].cpu(), want_grads=False)
        for key in ((0, 0), (1, 1)):
            assert rel_err(lat_c[key][:, j:j + 1], lat_o[key]) < 1e-10, (j, key)
        assert rel_err(recon[:, j:j + 1], recon_o) < 1e-10, j


@pytest.mark.gpu
def test_cfg4_batch1024_gradients_match_oracle_and_chunks(cfg4_run):
    """Gradients at full batch.  (a) The chamfer loss over the check jets S alone, with every kernel running over all 1024 jets:
    the parameter gradients against the oracle's gradients of the same loss on those jets (assert_grads_close).  (b) The
    gradient of the full-batch loss against the sum of the gradients of 128 chunks of 8 jets: a reduction that drops or
    repeats a partial row differs by the contribution of whole jets.  Bound, element by element: 2 n u sum_chunks |g_chunk|
    with n = B N^2 the longest sum (over edges).  sum_chunks |g_chunk| is at most the sum of |terms| the bound calls for, so
    elements whose chunk gradients cancel are held to 1e-2 of the tensor's largest such sum instead."""
    from lgn_autoencoder_b200 import fused
    from lgn_autoencoder_b200.train import training_step
    r = cfg4_run
    enc, dec, models, p4, p4n = r["enc"], r["dec"], r["models"], r["p4"], r["p4n"]
    S = r["jets"]
    idx = torch.tensor(S, device=_dev())
    _zero_grads(models)
    _, recon, _ = training_step(enc, dec, p4, l1_lambda=0.0, get_real="sum")
    fused.chamfer_loss(recon.index_select(1, idx), p4n.index_select(0, idx), "sum").backward()
    mine = _param_grads(models)
    ref = None
    for j in S:   # the loss is a sum over jets: the oracle one jet at a time
        _, _, _, g = _oracle(enc, dec, r["cfg"], p4n[j:j + 1].cpu())
        ref = g if ref is None else {kind: {k: (ref[kind][k] if g[kind][k] is None else g[kind][k] + ref[kind][k]) if ref[kind][k] is not None
                                            else g[kind][k] for k in g[kind]} for kind in g}
    for kind in ("enc", "dec"):
        assert_grads_close(mine[kind], {k: v for k, v in ref[kind].items() if v is not None})

    # (b) full batch against 128 chunks of 8 jets
    B, N = CFG4["B"], CFG4["N"]
    _zero_grads(models)
    loss, _, _ = training_step(enc, dec, p4, l1_lambda=0.0, get_real="sum")
    loss.backward()
    full = _param_grads(models)
    csum = {kind: {k: torch.zeros_like(v) for k, v in g.items()} for kind, g in full.items()}
    cabs = {kind: {k: torch.zeros_like(v) for k, v in g.items()} for kind, g in full.items()}
    for lo in range(0, B, 8):
        _zero_grads(models)
        l, _, _ = training_step(enc, dec, p4[lo:lo + 8], l1_lambda=0.0, get_real="sum")
        l.backward()
        for kind, g in _param_grads(models).items():
            for k, v in g.items():
                csum[kind][k] += v
                cabs[kind][k] += v.abs()
    n = B * N * N
    for kind in full:
        for k in full[kind]:
            scale = cabs[kind][k]
            scale = torch.maximum(scale, 1e-2 * scale.max())
            ratio = ((full[kind][k] - csum[kind][k]).abs() / (2 * n * U * scale + 1e-300)).max().item()
            assert ratio <= 1.0, (kind, k, ratio)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_composite_only_models_match_oracle(name):
    """Small batches of configurations the fused path refuses (max_zf 2, 9-16 channels, 17-20 radial basis functions) through
    the module API and autograd against the oracle: latent and reconstruction within 1e-10, loss, every parameter gradient
    (assert_grads_close)."""
    cfg = MODEL_CASES[name]
    dev = _dev()
    enc, dec = _build_model(cfg, dev)
    assert not enc.fused, name   # (the decoder's radial functions see masked edges only: it may take more basis functions fused)
    from lgn_autoencoder_b200 import fused
    from oracle import lgae_oracle as orc
    data = orc.synthetic_jets(cfg["batch"], cfg["n"], seed=cfg["seed"] + 1, mass_scale=0.05)
    pn, _ = orc.normalize_p4_overall_max(data["p4"])
    lat_o, recon_o, loss_o, g_o = _oracle(enc, dec, cfg, pn)
    models = {"enc": enc, "dec": dec}
    _zero_grads(models)
    p4 = pn.to(dev)
    latent = enc({"p4": p4})
    recon = dec(latent)
    loss = fused.chamfer_loss(recon, p4, "sum")
    loss.backward()
    for key in ((0, 0), (1, 1)):
        assert rel_err(latent[key], lat_o[key]) < 1e-10, (name, key)
    assert rel_err(recon, recon_o) < 1e-10, name
    assert abs(loss.item() - loss_o.item()) <= 1e-10 * abs(loss_o.item()), name
    mine = _param_grads(models)
    for kind in ("enc", "dec"):
        assert_grads_close(mine[kind], {k: v for k, v in g_o[kind].items() if v is not None})
