"""CPU tests of the fp64 reference for the importance-weighted log-likelihood (tests/iw_ref.py): the logmeanexp's properties
and NaN / inf rules, and the port-side estimator on a tiny fixture."""
import math

import torch

from flowcompare_b200 import configs
from oracle import port
from oracle.make_golden import fixture_inputs
from tests.iw_ref import logmeanexp, port_log_prob_iw

torch.set_grad_enabled(False)
INF, NAN = float("inf"), float("nan")


def test_identical_draws_give_the_single_value():
    v = torch.tensor([-3.25, 0.0, 17.5, -1234.5], dtype=torch.float64)
    for K in (1, 2, 7, 64):
        got = logmeanexp(v.expand(K, -1))
        assert (got - v).abs().max().item() < 1e-12


def test_iw_is_at_least_the_mean_of_its_draws():
    g = torch.Generator().manual_seed(3)
    d = torch.randn(16, 5000, generator=g, dtype=torch.float64) * 40 - 300
    iw = logmeanexp(d)
    assert (iw >= d.mean(0) - 1e-9).all()
    assert (iw <= d.max(0).values + 1e-9).all()          # and never above the best draw
    # K = 1 is the draw itself
    assert torch.equal(logmeanexp(d[:1]), d[0])


def test_matches_direct_formula_where_it_does_not_overflow():
    d = torch.tensor([[-1.0, 2.0], [0.5, 3.0], [-2.0, -4.0]], dtype=torch.float64)
    want = torch.log(torch.exp(d).mean(0))
    assert (logmeanexp(d) - want).abs().max().item() < 1e-14
    # far below exp's range: the max shift keeps it finite
    assert abs(logmeanexp(d - 5000.0)[0].item() - (want[0].item() - 5000.0)) < 1e-9


def test_nan_and_inf_rules():
    cols = {
        "nan": [1.0, NAN, 2.0],
        "nan_beats_inf": [INF, NAN, 2.0],
        "pinf": [1.0, INF, -INF],
        "all_ninf": [-INF, -INF, -INF],
        "ninf_drops_out": [-INF, 0.0, -INF],
    }
    d = torch.tensor(list(cols.values()), dtype=torch.float64).T
    got = dict(zip(cols, logmeanexp(d).tolist()))
    assert math.isnan(got["nan"]) and math.isnan(got["nan_beats_inf"])
    assert got["pinf"] == INF
    assert got["all_ninf"] == -INF
    assert abs(got["ninf_drops_out"] - (0.0 - math.log(3))) < 1e-15


def test_port_iw_on_a_tiny_fixture():
    """K = 1 is port.flow_log_prob itself; K copies of one draw give that draw; distinct draws give IW >= their mean."""
    cfg, fsd, esd, batch = fixture_inputs("tiny_dgcnn_attn")
    x = batch["extract_1"][:1, :24]
    ctx = torch.randn(1, 40, configs.derive(cfg)["input_embedding_dim"], generator=torch.Generator().manual_seed(5))
    S = configs.derive(cfg)["latent_dim"] - configs.derive(cfg)["input_dim"]
    eps = torch.randn(3, 1, 24, S, generator=torch.Generator().manual_seed(6))
    iw1, d1 = port_log_prob_iw(cfg, fsd, x, ctx, None, eps[:1])
    want = port.flow_log_prob(port.to_dtype(fsd, torch.float64), configs.derive(cfg), x.double()[..., :6], ctx.double(), None,
                              eps[0].double())
    assert torch.equal(d1[0], want) and torch.equal(iw1, want)
    iw_same, _ = port_log_prob_iw(cfg, fsd, x, ctx, None, eps[:1].expand(4, -1, -1, -1))
    assert (iw_same - want).abs().max().item() < 1e-9
    iw3, d3 = port_log_prob_iw(cfg, fsd, x, ctx, None, eps)
    assert d3.shape == (3, 1, 24) and (iw3 >= d3.mean(0) - 1e-9).all()
    assert (d3[0] != d3[1]).any()                      # the draws really differ


def test_port_iw_takes_cif_draws_per_draw():
    cfg, fsd, esd, batch = fixture_inputs("a18_cif")
    dcfg = configs.derive(cfg)
    x, E = batch["extract_1"][:1, :16], dcfg["input_embedding_dim"]
    ctx = torch.randn(1, 32, E, generator=torch.Generator().manual_seed(8))
    S, Sc, L = dcfg["latent_dim"] - dcfg["input_dim"], dcfg["cif_latent_dim"] - dcfg["latent_dim"], dcfg["n_flow_layers"]
    g = torch.Generator().manual_seed(9)
    eps, eps_cif = torch.randn(2, 1, 16, S, generator=g), torch.randn(2, L, 1, 16, Sc, generator=g)
    _, d = port_log_prob_iw(cfg, fsd, x, ctx, None, eps, eps_cif)
    want = port.flow_log_prob(port.to_dtype(fsd, torch.float64), dcfg, x.double()[..., :6], ctx.double(), None, eps[1].double(),
                              eps_cif=eps_cif[1].double())
    assert torch.equal(d[1], want)
