"""CPU tests of the fp64 reference of the attention score gradients (tests/attention_score_grads_ref.py): the recorder leaves the
port's log-prob unchanged, its retained d lp_i / d s_ij matches central differences of lp_i under a bias on the scores, equals the
closed form P (dO.v - dO.o) the CUDA kernel evaluates, and every row sums to zero."""
import pytest
import torch

from flowcompare_b200 import configs, packing
from oracle import port
from oracle.make_golden import fixture_inputs
from tests.attention_score_grads_ref import closed_form, port_score_grads, score_grads


def _inputs(name, n_points, n_ctx, seed):
    cfg, fsd, esd, batch = fixture_inputs(name)
    dcfg = configs.derive(cfg)
    g = torch.Generator().manual_seed(seed)
    B = 2
    x = batch["extract_1"][:B, :n_points, :dcfg["input_dim"]].double()
    ctx = torch.randn(B, n_ctx, dcfg["input_embedding_dim"], generator=g)
    extra = torch.randn(B, 1, generator=g) if dcfg["using_extra_context"] else None
    eps = torch.randn(B, n_points, dcfg["latent_dim"] - dcfg["input_dim"], generator=g)
    return cfg, fsd, x, ctx, extra, eps


@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "a18_identity_augmenter"])
def test_recorder_leaves_log_prob_unchanged(monkeypatch, name):
    cfg, fsd, x, ctx, extra, eps = _inputs(name, 12, 40, seed=1)
    dcfg = configs.derive(cfg)
    ex = None if extra is None else extra.double().unsqueeze(1).expand(-1, x.shape[1], -1)
    eps = eps.double() if dcfg["latent_dim"] > dcfg["input_dim"] else None
    want = port.flow_log_prob(port.to_dtype(fsd, torch.float64), dcfg, x, ctx.double(), ex, eps)
    lp, rec = port_score_grads(monkeypatch, cfg, fsd, x, ctx, extra, eps)
    assert torch.equal(lp, want)
    assert port.cross_attention.__name__ == "cross_attention" and port.cross_attention.__module__ == "oracle.port"
    assert list(rec) == packing.attention_block_names(cfg)
    for g in score_grads(rec).values():
        assert g is not None and g.shape == (x.shape[0], x.shape[1], ctx.shape[1])


def test_score_gradient_matches_central_differences(monkeypatch):
    """A bias h on column j of one block's scores moves every lp_i by h * d lp_i / d s_ij (rows are independent), so one pair of
    runs checks a whole column; two columns of every block."""
    cfg, fsd, x, ctx, extra, eps = _inputs("tiny_dgcnn_attn", 6, 24, seed=3)
    _, rec = port_score_grads(monkeypatch, cfg, fsd, x, ctx, extra, eps)
    grads = score_grads(rec)
    h = 1e-5
    worst = 0.0
    for prefix, g in grads.items():
        for j in (0, 17):
            lp_p, _ = port_score_grads(monkeypatch, cfg, fsd, x, ctx, extra, eps, bias=(prefix, j, h), backward=False)
            lp_m, _ = port_score_grads(monkeypatch, cfg, fsd, x, ctx, extra, eps, bias=(prefix, j, -h), backward=False)
            fd = (lp_p - lp_m) / (2 * h)
            err = ((fd - g[..., j]).abs() / g.abs().amax(-1)).max().item()
            worst = max(worst, err)
            assert err < 1e-6, (prefix, j, err)
    print(f"max |fd - sim.grad| / row max {worst:.3e}")


@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "a18_permute_relu"])
def test_closed_form_and_zero_row_sums(monkeypatch, name):
    cfg, fsd, x, ctx, extra, eps = _inputs(name, 10, 33, seed=2)
    _, rec = port_score_grads(monkeypatch, cfg, fsd, x, ctx, extra, eps)
    for prefix, r in rec.items():
        g = r["sim"].grad
        scale = g.abs().amax(-1, keepdim=True)
        assert ((closed_form(r) - g).abs() / scale).max().item() < 1e-12, prefix
        assert (g.sum(-1).abs() / scale[..., 0]).max().item() < 1e-12, prefix
