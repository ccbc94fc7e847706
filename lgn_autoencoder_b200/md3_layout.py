"""Algebra of one maxdim-3 LGN level (max_zf = 1) as the fused forward kernels evaluate it (csrc/lgae_md3.cu).

A node carries the irreps (0,0), (1,1), (2,0), (0,2), (2,2): 20 complex components per channel, stored in that order
(``IRREPS`` / ``COMP_OFFSET``).  The level output of irrep tau, channel c' is

    out_tau[c'] = sum_col W_tau[c', col] cat_tau[col],   cat_tau = [ag pieces | node | sq pieces], C channels per piece,

where the pieces and their order are those of the layer-level composite: ``cg_product`` loops over the keys of its first
operand, then of its second (oracle ``cg_product``), ``cat_reps`` concatenates [ag, node, sq], and the node's own key order is
the set order in which ``MixReps`` emits its parts, with (0,0) moved to the end by the scalar MLP.  Everything here is
derived from ``CGDict(maxdim=3)`` and those rules; ``tools/gen_md3_tables.py`` writes it as ``csrc/lgae_md3_tables.h``.

Piece kinds (what a term (x, y, coef) of output component m multiplies):
    NODE  z[off(tau) + m]                                     (no terms)
    AG0   (1+i) sum coef * S0[x]     S0[a]   = sum_j R0_ij z_j[a]               (edge (0,0) = R0 (1+i))
    AG1   sum coef * T[x]            T[4a+d] = sum_j R1_ij z_j[a] Y_ij[d]        (edge (1,1) = R1 canon(p_i - p_j))
    SQ    sum coef * z[x] * z[y]                                                 (self product)
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

Key = Tuple[int, int]

MAXDIM = 3
IRREPS: Tuple[Key, ...] = ((0, 0), (1, 1), (2, 0), (0, 2), (2, 2))
DIM = {k: (k[0] + 1) * (k[1] + 1) for k in IRREPS}
COMP_OFFSET = {(0, 0): 0, (1, 1): 1, (2, 0): 5, (0, 2): 8, (2, 2): 11}
N_COMP = 20
EDGE_ORDER: Tuple[Key, ...] = ((0, 0), (1, 1))   # rad_funcs / zonal parts, l = 0 .. max_zf
KIND_NODE, KIND_AG0, KIND_AG1, KIND_SQ = 0, 1, 2, 3
# node key orders the kernels know: level 0 (input map: (0,0), (1,1) only), later levels with and without the scalar MLP
VARIANTS = ("level0", "mlp", "nomlp")
COEF_EPS = 1e-13


def set_order(keys: Sequence[Key]) -> List[Key]:
    """The order in which a MixReps emits its parts (``GWeightDict.keys()``: the iteration order of a set)."""
    return list(set(keys))


def node_order(variant: str) -> List[Key]:
    if variant == "level0":
        return set_order([(0, 0), (1, 1)])
    order = set_order(IRREPS)
    if variant == "mlp":   # CGMLP pops (0,0) and re-inserts it
        order = [k for k in order if k != (0, 0)] + [(0, 0)]
    return order


def product_keys(k1: Key, k2: Key, maxdim: int = MAXDIM) -> List[Key]:
    """Output irreps of one (k1, k2) pair in cg_product's order."""
    return [(k, n) for k in range(abs(k1[0] - k2[0]), min(maxdim, k1[0] + k2[0] + 1), 2)
            for n in range(abs(k1[1] - k2[1]), min(maxdim, k1[1] + k2[1] + 1), 2)]


def blocks(order: Sequence[Key]) -> Dict[Key, List[Tuple[int, Key, Key]]]:
    """Per output irrep (in IRREPS order): the cat pieces (kind, rep1, rep2) in column order, C columns each."""
    out: Dict[Key, List[Tuple[int, Key, Key]]] = {t: [] for t in IRREPS}
    for r in order:                       # ag = cg_product(node, edge, aggregate=True)
        for e in EDGE_ORDER:
            for t in product_keys(r, e):
                out[t].append((KIND_AG0 if e == (0, 0) else KIND_AG1, r, e))
    for r in order:                       # node
        out[r].append((KIND_NODE, r, r))
    for r1 in order:                      # sq = cg_product(node, node)
        for r2 in order:
            for t in product_keys(r1, r2):
                out[t].append((KIND_SQ, r1, r2))
    return out


def piece_terms(cg, kind: int, r1: Key, r2: Key, tau: Key) -> List[List[Tuple[int, int, float]]]:
    """Per output component m of tau: the terms (x, y, coef) of one piece, in the order of the composite's matmul."""
    if kind == KIND_NODE:
        return [[] for _ in range(DIM[tau])]
    mat = cg[(r1, r2)][tau]                     # (d_tau, d1 * d2)
    d2 = DIM[r2]
    terms = []
    for m in range(DIM[tau]):
        row = []
        for col in range(mat.shape[1]):
            c = float(mat[m, col])
            if abs(c) <= COEF_EPS:
                continue
            a, b = divmod(col, d2)
            xa = COMP_OFFSET[r1] + a
            if kind == KIND_AG0:
                row.append((xa, 0, c))
            elif kind == KIND_AG1:
                row.append((4 * xa + b, 0, c))
            else:
                row.append((xa, COMP_OFFSET[r2] + b, c))
        terms.append(row)
    return terms


def tables(cg):
    """Everything the kernels read: unique pieces with their term ranges, and per (variant, tau) the piece ids in column order."""
    pieces: List[Tuple[int, Key, Key, Key]] = []
    index: Dict[Tuple[int, Key, Key, Key], int] = {}
    var_blocks: Dict[str, Dict[Key, List[int]]] = {}
    for v in VARIANTS:
        bl = blocks(node_order(v))
        var_blocks[v] = {}
        for t in IRREPS:
            ids = []
            for kind, r1, r2 in bl[t]:
                key = (kind, r1, r2, t)
                if key not in index:
                    index[key] = len(pieces)
                    pieces.append(key)
                ids.append(index[key])
            var_blocks[v][t] = ids
    ranges: List[int] = []
    terms: List[Tuple[int, int, float]] = []
    first: List[int] = []
    for kind, r1, r2, t in pieces:
        first.append(len(ranges))
        for row in piece_terms(cg, kind, r1, r2, t):
            ranges.append(len(terms))
            terms.extend(row)
    ranges.append(len(terms))
    return pieces, first, ranges, terms, var_blocks


def mix_columns(variant: str) -> Dict[Key, int]:
    """Number of C-channel pieces in each irrep's concatenation (the mix weights are (2, C', n * C))."""
    bl = blocks(node_order(variant))
    return {t: len(bl[t]) for t in IRREPS}
