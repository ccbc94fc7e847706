"""The maxdim-3 forward count of flop_model follows the counting rule of the maxdim-2 constants (SURVEY.md section 8(d)): a CG
product counts once if it has a non-zero coefficient in an allowed output.  No GPU needed."""


def test_rule_reproduces_the_maxdim2_constant():
    from lgn_autoencoder_b200 import flop_model as F
    agg, _ = F.cg_counts([(0, 0), (1, 1)], 2)
    assert agg == F._AGG_PER_EDGE_CH == 150


def test_cfg4_forward_count():
    """cfg-4 (enc 6-6-8-8 / dec 8-8-6-6, K = 20, MLP 6 x 6) at N = 30: SURVEY section 8(d)'s 66.1 MFLOP per jet."""
    from lgn_autoencoder_b200 import flop_model as F
    total = sum(F.md3_forward_flops_per_jet(30, [6, 6, 8, 8], [8, 8, 6, 6]).values()) / 1e6
    assert abs(total - 66.1) < 0.05, total


def test_maxdim2_counts_unchanged():
    from lgn_autoencoder_b200 import flop_model as F
    assert abs(F.step_flops_per_jet(30, [3, 3, 4, 4], [4, 4, 3, 3], backward=False) / 1e6 - 9.13908) < 1e-5
