"""Reference-faithful algorithmic FLOP counts of the LGAE hot path (SURVEY.md section 8(d)): the numerator of every
roofline figure in bench.py.  Real flops only: complex mul = 6, complex add = 2, complex x real-coefficient MAC = 4,
reciprocal / sqrt / div = 1, only non-zero CG coefficients.  The counts describe the REFERENCE's algorithm
(O(N^2) decoder aggregation, full radial functions in every level); algebraic savings made by the kernels do not
shrink them."""
from __future__ import annotations

from typing import Dict, List

# maxdim-2 CG bookkeeping for a level with node irreps {(0,0),(1,1)} x edge irreps {(0,0),(1,1)}:
#   products: S.e0 (1 comp), V.e0 (4), S.e1 (4), V.e1 -> (0,0) (1 comp from 4 products)
_D_EDGE = 5            # sum_l d_l of the zonal functions (1 + 4)
_AGG_PER_EDGE_CH = 150  # 6*#products + 4*nnz + 2*sum(out comps), SURVEY 8(d)
_POW_PER_NODE_CH = 6 * 10 + 4 * 14   # self product: same structure without the neighbour sum


def level_flops(n: int, c_in: int, c_out: int, k_basis: int, encoder: bool, mlp_width: int, mlp_hidden: int) -> Dict[str, float]:
    """Forward flops of one LGN level for one jet, split by stage."""
    out = {}
    out["radial"] = n * n * (6 * k_basis + 2 * k_basis * 2 * c_in * 2) if encoder else 0.0
    out["edge"] = n * n * c_in * 6 * _D_EDGE
    out["aggregate"] = n * n * c_in * _AGG_PER_EDGE_CH
    out["power"] = n * c_in * _POW_PER_NODE_CH
    out["mix"] = n * 8 * (1 + 4) * c_out * 5 * c_in
    w = mlp_width
    out["mlp"] = n * 2 * (2 * c_out * w + (mlp_hidden - 1) * w * w + w * 2 * c_out) if mlp_hidden else 0.0
    return out


def model_flops(n: int, channels: List[int], k_basis: int, encoder: bool, mlp_width_mul: int, mlp_hidden: int) -> Dict[str, float]:
    tot: Dict[str, float] = {}
    for l in range(len(channels) - 1):
        lf = level_flops(n, channels[l], channels[l + 1], k_basis, encoder, mlp_width_mul * 2 * channels[l + 1], mlp_hidden)
        for k, v in lf.items():
            tot[k] = tot.get(k, 0.0) + v
    return tot


def step_flops_per_jet(n: int, enc_channels: List[int], dec_channels: List[int], num_basis_fn: int = 10, mlp_width_mul: int = 6,
                       mlp_hidden: int = 6, backward: bool = True) -> float:
    """Encoder + decoder forward (x3 with the backward pass, SURVEY 8(d))."""
    e = model_flops(n, enc_channels, 2 * num_basis_fn, True, mlp_width_mul, mlp_hidden)
    d = model_flops(n, dec_channels, 2 * num_basis_fn, False, mlp_width_mul, mlp_hidden)
    fwd = sum(e.values()) + sum(d.values())
    return fwd * (3.0 if backward else 1.0)


# ---- maxdim 3 (forward only): node irreps (0,0), (1,1), (2,0), (0,2), (2,2); level 0 has (0,0), (1,1) ----------------------
def _pair_counts(cg, r1, r2, maxdim: int):
    """(#products, nnz, sum of output dims) of one channel-wise CG product r1 (x) r2 with outputs below ``maxdim``.  A product
    z1[a] z2[b] counts once if it has a non-zero coefficient in at least one allowed output (the rule of the maxdim-2 constants:
    V.e1 -> (0,0) is 4 products, not 16)."""
    from . import md3_layout as M
    outs = M.product_keys(r1, r2, maxdim)
    used = None
    nnz = 0
    for t in outs:
        nzm = cg[(r1, r2)][t].abs() > M.COEF_EPS          # (d_out, d1 * d2)
        nnz += int(nzm.sum())
        used = nzm.any(0) if used is None else (used | nzm.any(0))
    return (int(used.sum()) if used is not None else 0), nnz, sum(M.DIM[t] for t in outs)


def cg_counts(node_keys, maxdim: int):
    """(aggregate per edge and channel, self product per node and channel) of a level whose nodes carry ``node_keys``, edges
    (0,0) and (1,1): 6 #products + 4 nnz + 2 sum(out comps), and 6 #products + 4 nnz.  cg_counts([(0,0), (1,1)], 2)[0] == 150 ==
    _AGG_PER_EDGE_CH."""
    from . import md3_layout as M
    from .cg_lib import CGDict
    cg = CGDict(maxdim=max(maxdim, 2))
    agg = sum(6 * p + 4 * z + 2 * o for p, z, o in (_pair_counts(cg, r, e, maxdim) for r in node_keys for e in M.EDGE_ORDER))
    pw = sum(6 * p + 4 * z for p, z, _ in (_pair_counts(cg, r1, r2, maxdim) for r1 in node_keys for r2 in node_keys))
    return agg, pw


def _md3_cg_counts(variant: str):
    """(aggregate per edge and channel, self product per node and channel, mix complex MACs per (c_in, c_out)) of one maxdim-3 level,
    counted as above from the non-zero CG coefficients of CGDict(maxdim=3)."""
    from . import md3_layout as M
    agg, pw = cg_counts(M.node_order(variant), M.MAXDIM)
    cols = M.mix_columns(variant)
    mix = sum(M.DIM[t] * cols[t] for t in M.IRREPS)
    return agg, pw, mix


def md3_level_flops(n: int, level: int, c_in: int, c_out: int, k_basis: int, encoder: bool, mlp_width: int, mlp_hidden: int,
                    mlp: bool = True) -> Dict[str, float]:
    """Forward flops of one maxdim-3 LGN level for one jet, split by stage (the reference's algorithm, as level_flops)."""
    agg, pw, mix = _md3_cg_counts("level0" if level == 0 else ("mlp" if mlp else "nomlp"))
    out = {}
    out["radial"] = n * n * (6 * k_basis + 2 * k_basis * 2 * c_in * 2) if encoder else 0.0
    out["edge"] = n * n * c_in * 6 * _D_EDGE
    out["aggregate"] = n * n * c_in * agg
    out["power"] = n * c_in * pw
    out["mix"] = n * 8 * mix * c_out * c_in
    w = mlp_width
    out["mlp"] = n * 2 * (2 * c_out * w + (mlp_hidden - 1) * w * w + w * 2 * c_out) if mlp_hidden else 0.0
    return out


def md3_forward_flops_per_jet(n: int, enc_channels: List[int], dec_channels: List[int], num_basis_fn: int = 10, mlp_width_mul: int = 6,
                              mlp_hidden: int = 6) -> Dict[str, float]:
    """Encoder + decoder forward of a maxdim-3 model for one jet, by stage."""
    tot: Dict[str, float] = {}
    for chans, enc in ((enc_channels, True), (dec_channels, False)):
        for l in range(len(chans) - 1):
            lf = md3_level_flops(n, l, chans[l], chans[l + 1], 2 * num_basis_fn, enc, mlp_width_mul * 2 * chans[l + 1], mlp_hidden)
            for k, v in lf.items():
                tot[k] = tot.get(k, 0.0) + v
    return tot
