"""CPU tests of the input-gradient pass's references and packing: the fp64 port's autograd gradient (tests/grad_ref.py) against
central finite differences, and packing.pack_flow_grad's transposed Linears against the folded forward matrices they stand for."""
import pytest
import torch

from flowcompare_b200 import configs, packing
from oracle import port
from oracle.make_golden import fixture_inputs
from tests.grad_ref import dense_linear, forward_linears, grad_linears, port_log_prob_grad


def _inputs(name, n_points, n_ctx, seed):
    cfg, fsd, esd, batch = fixture_inputs(name)
    dcfg = configs.derive(cfg)
    g = torch.Generator().manual_seed(seed)
    B = 1
    x = batch["extract_1"][:B, :n_points, :dcfg["input_dim"]].double()
    E = dcfg["input_embedding_dim"]
    ctx = torch.randn(B, E, generator=g) if dcfg["global"] else torch.randn(B, n_ctx, E, generator=g)
    extra = torch.randn(B, 1, generator=g) if dcfg["using_extra_context"] else None
    eps = torch.randn(B, n_points, dcfg["latent_dim"] - dcfg["input_dim"], generator=g)
    return cfg, fsd, x, ctx, extra, eps


@pytest.mark.parametrize("name,n_points,n_ctx", [("tiny_dgcnn_attn", 5, 40), ("tiny_dgcnn_global", 4, 1),
                                                 ("tiny_dgcnn_attn_extra", 4, 24), ("full_dgcnn_attn", 2, 48)])
def test_port_gradient_matches_central_differences(name, n_points, n_ctx):
    """Points are scored independently, so one coordinate can be perturbed in every point at once."""
    cfg, fsd, x, ctx, extra, eps = _inputs(name, n_points, n_ctx, seed=3)
    _, g = port_log_prob_grad(cfg, fsd, x, ctx, extra, eps)
    h = 1e-6
    for c in range(x.shape[-1]):
        xp, xm = x.clone(), x.clone()
        xp[..., c] += h
        xm[..., c] -= h
        fd = (port_log_prob_grad(cfg, fsd, xp, ctx, extra, eps)[0] - port_log_prob_grad(cfg, fsd, xm, ctx, extra, eps)[0]) / (2 * h)
        err = ((fd - g[..., c]).abs() / g.abs().amax(-1).clamp_min(1.0)).max().item()
        assert err < 1e-6, (name, c, err)


def test_gradient_of_a_weighted_sum():
    cfg, fsd, x, ctx, extra, eps = _inputs("tiny_dgcnn_attn", 6, 32, seed=4)
    _, g = port_log_prob_grad(cfg, fsd, x, ctx, extra, eps)
    w = torch.randn(x.shape[:2], dtype=torch.float64, generator=torch.Generator().manual_seed(5))
    xv = x.clone().requires_grad_(True)
    with torch.enable_grad():
        lp = port.flow_log_prob(port.to_dtype(fsd, torch.float64), configs.derive(cfg), xv, ctx.double(), None, eps.double())
        (gw,) = torch.autograd.grad((w * lp).sum(), xv)
    assert (gw - w[..., None] * g).abs().max().item() < 1e-12


@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "tiny_dgcnn_global", "a18_permute_relu",
                                  "a18_fullcombiner_noactnorm", "a18_expcombiner_global", "a18_identity_augmenter"])
def test_grad_arena_holds_the_transposed_forward_matrices(name):
    cfg, fsd, esd, batch = fixture_inputs(name)
    fh, ft, fa = packing.pack_flow(fsd, cfg)
    gh, gt, ga = packing.pack_flow_grad(fsd, cfg)
    fwd, grd = forward_linears(fh, ft), grad_linears(fh, gt)
    inner = 64
    checked = 0
    for key, (off, K1, K2, N) in fwd.items():
        if key.endswith(".kv"):
            continue                                   # no gradient flows to the context
        W = dense_linear(fa, off, K1, K2, N)
        block, layer = key.rsplit(".", 1)
        if layer == "in":
            k_x = K1
            Wx = dense_linear(ga, *grd[f"{block}.in_x"])
            assert torch.equal(Wx.t(), W[:, :k_x]), key
            if K2:
                assert K2 == inner
                assert torch.equal(dense_linear(ga, *grd[f"{block}.in_o"]).t(), W[:, k_x:]), key
        else:
            assert torch.equal(dense_linear(ga, *grd[key]).t(), W), key
        checked += 1
    assert checked == len([k for k in fwd if not k.endswith(".kv")])
    assert int(gh[0]) == packing.GRAD_MAGIC and int(gh[1]) == packing.ARENA_VERSION


@pytest.mark.parametrize("name,what", [("a18_spline", "RationalQuadraticSplineCoupling"), ("a18_expo", "ExponentialCoupling"),
                                       ("a18_cif", "CIFblock")])
def test_unsupported_flows_are_named(name, what):
    cfg, fsd, esd, batch = fixture_inputs(name)
    assert packing.grad_unsupported_transform(cfg) == what
    with pytest.raises(NotImplementedError, match=what):
        packing.pack_flow_grad(fsd, cfg)
