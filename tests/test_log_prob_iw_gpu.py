"""GPU tests of the multi-draw log-likelihood (engine.log_prob_iw -> fc_flow_log_prob_draws + fc_logmeanexp): every draw is
bitwise the single-draw log_prob, the estimate matches the fp64 port, the reduction follows its rules, the result does not
depend on the batch or the pass split (also at the 2^20-row pass cap), the consumers (change maps, evaluation) use it, and the
points of a cloud are scored independently (the K*N row layout rests on that)."""
import math

import pytest
import torch

from flowcompare_b200 import configs, engine as eng, lib as fclib, spec
from oracle.make_golden import fixture_inputs
from tests.iw_ref import logmeanexp, port_log_prob_iw

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
DEV = "cuda:0"
PRECISIONS = ["fp32", "tf32x3", "fp16x3"]
INF, NAN = float("inf"), float("nan")


def _setup(name, precision="fp32"):
    cfg, fsd, esd, batch = fixture_inputs(name)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    ctx = e.embed(batch["extract_0"].to(DEV))
    extra = batch["extra_context"]
    return cfg, fsd, batch, e, ctx, None if extra is None else extra.to(DEV)


def _draws(e, K, B, N, seed):
    g = torch.Generator().manual_seed(seed)
    eps = torch.randn(K, B, N, e.D - e.d_in, generator=g).to(DEV)
    eps_cif = torch.randn(K, e.L, B, N, e.cif_S, generator=g).to(DEV) if e.cif_S else None
    return eps, eps_cif


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "tiny_dgcnn_global", "tiny_paconv_attn",
                                  "mid_dgcnn_attn", "a18_spline", "a18_expo", "a18_cif"])
def test_each_draw_is_log_prob(name, precision):
    cfg, fsd, batch, e, ctx, extra = _setup(name, precision)
    x = batch["extract_1"].to(DEV)
    B, N, K = x.shape[0], x.shape[1], 3
    eps, eps_cif = _draws(e, K, B, N, seed=1)
    iw, draws = e.log_prob_iw(x, ctx, extra, n_draws=K, eps=eps, eps_cif=eps_cif, return_draws=True)
    assert draws.shape == (K, B, N) and iw.shape == (B, N)
    for k in range(K):
        lp = e.log_prob(x, ctx, extra, eps=eps[k], eps_cif=None if eps_cif is None else eps_cif[k])
        assert torch.equal(draws[k], lp), (k, (draws[k] - lp).abs().max().item())
    assert not torch.equal(draws[0], draws[1])
    assert torch.isfinite(iw).all() and (iw.double() >= draws.double().mean(0) - 1e-3).all()
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "tiny_dgcnn_global", "tiny_paconv_attn"])
def test_iw_matches_fp64_port(name, precision):
    cfg, fsd, batch, e, ctx, extra = _setup(name, precision)
    x = batch["extract_1"].to(DEV)
    eps, _ = _draws(e, 4, x.shape[0], x.shape[1], seed=2)
    iw = e.log_prob_iw(x, ctx, extra, n_draws=4, eps=eps)
    want, _ = port_log_prob_iw(cfg, fsd, x, ctx, extra, eps)
    err = (iw.cpu().double() - want).abs().max().item()
    print(f"{name} {precision}: max |IW - fp64 port IW| = {err:.3e}")
    assert err < 1e-3
    e.close()


def _lme(draws):
    lib = fclib.load()
    d = draws.to(DEV, torch.float32).contiguous()
    out = torch.empty(d.shape[1:], dtype=torch.float32, device=DEV)
    fclib.check(lib.fc_logmeanexp(d.data_ptr(), d.shape[0], out.numel(), out.data_ptr(), torch.cuda.current_stream().cuda_stream),
                "fc_logmeanexp")
    return out


def test_logmeanexp_against_fp64():
    g = torch.Generator().manual_seed(4)
    for K, M in ((1, 1000), (5, 10007), (37, 4099), (256, 3000)):
        d = torch.randn(K, M, generator=g) * torch.rand(1, M, generator=g) * 60 - 400 * torch.rand(1, M, generator=g)
        got = _lme(d).cpu().double()
        want = logmeanexp(d)
        rel = (got - want).abs() / want.abs().clamp_min(1.0)       # relative, floored at one nat
        assert rel.max().item() <= 1e-6, (K, rel.max().item())
    v = torch.tensor([-3.25, 0.0, 17.5, -1234.5, 1e-30, 88.0])
    for K in (1, 3, 16, 100):      # K equal draws give that value exactly
        assert torch.equal(_lme(v.expand(K, -1)).cpu(), v)


def test_logmeanexp_nan_and_inf_rules():
    cols = [[1.0, NAN, 2.0], [INF, NAN, 2.0], [NAN, -INF, -INF], [1.0, INF, -INF], [INF, INF, INF], [-INF, -INF, -INF],
            [-INF, 0.0, -INF], [-INF, -5.0, 3.0]]
    d = torch.tensor(cols, dtype=torch.float32).T
    got, want = _lme(d).cpu().double(), logmeanexp(d)
    assert torch.equal(torch.isnan(got), torch.isnan(want)) and torch.isnan(got[:3]).all()
    inf = torch.isinf(want)
    assert torch.equal(torch.isinf(got), inf) and torch.equal(got[inf], want[inf])
    assert got[3] == INF and got[4] == INF and got[5] == -INF
    assert abs(got[6] - (-math.log(3))) < 1e-6 and abs(got[7] - want[7]) <= 1e-6 * abs(want[7])


@pytest.mark.parametrize("precision", PRECISIONS)
def test_invariant_run_to_run_batch_and_pass_split(precision):
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn", precision)
    x = batch["extract_1"].to(DEV)
    B, N, K = x.shape[0], x.shape[1], 16
    eps, _ = _draws(e, K, B, N, seed=5)
    iw, d = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, return_draws=True)
    for _ in range(2):
        iw2, d2 = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, return_draws=True)
        assert torch.equal(iw, iw2) and torch.equal(d, d2)
    iw1, d1 = e.log_prob_iw(x[1:2], ctx[1:2], n_draws=K, eps=eps[:, 1:2].contiguous(), return_draws=True)
    assert torch.equal(iw1[0], iw[1]) and torch.equal(d1[:, 0], d[:, 1])      # one cloud alone vs inside the batch
    iw3, d3 = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, return_draws=True, draws_per_pass=3)
    assert torch.equal(iw3, iw) and torch.equal(d3, d)
    # a workspace budget that allows one draw per pass
    budget = e.lib.fc_flow_log_prob_draws_workspace_bytes(e._flow["handle"], B, N, ctx.shape[1], 1)
    iw4 = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, workspace_budget=budget)
    assert torch.equal(iw4, iw)
    # ... and one that allows one cloud and one draw per pass
    budget = e.lib.fc_flow_log_prob_draws_workspace_bytes(e._flow["handle"], 1, N, ctx.shape[1], 1)
    iw5, d5 = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, workspace_budget=budget, return_draws=True)
    assert torch.equal(iw5, iw) and torch.equal(d5, d)
    e.close()


def test_one_pass_at_the_row_cap():
    """K*B*N = 2^20 rows in one pass (1.2 GB of eps, ~8 GB of workspace) equals the same draws in passes of 3000 draws."""
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn", "fp16x3")
    x = batch["extract_1"][:, :64].to(DEV)
    B, N = x.shape[0], x.shape[1]
    K = eng.IW_MAX_PASS_ROWS // (B * N)
    assert K * B * N == 1 << 20
    eps = torch.randn(K, B, N, e.D - e.d_in, device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))
    iw, d = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, return_draws=True)
    iw_s, d_s = e.log_prob_iw(x, ctx, n_draws=K, eps=eps, return_draws=True, draws_per_pass=3000)
    assert torch.equal(d, d_s) and torch.equal(iw, iw_s)
    for k in (0, K // 2, K - 1):
        assert torch.equal(d[k], e.log_prob(x, ctx, eps=eps[k]))
    assert torch.isfinite(iw).all()
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_deterministic_flow_iw_is_log_prob(precision):
    cfg, fsd, batch, e, ctx, extra = _setup("a18_identity_augmenter", precision)
    x = batch["extract_1"].to(DEV)
    lp = e.log_prob(x, ctx, extra, eps=batch["eps"].to(DEV))      # eps [B, N, 0]: there is nothing to draw
    iw, d = e.log_prob_iw(x, ctx, extra, n_draws=5, return_draws=True)
    assert torch.equal(iw, lp)
    assert all(torch.equal(d[k], lp) for k in range(5))
    e.close()


def _four_batches(cfg, B):
    out = []
    for i in range(4):
        b = spec.synthetic_batch(cfg, B, seed=60 + i)
        out.append((b["extract_0"].to(DEV), b["extract_1"].to(DEV), None if b["extra_context"] is None else b["extra_context"].to(DEV)))
    return out


def test_change_maps_with_draws():
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn_extra", "tf32x3")
    B, K = 2, 4
    batches = _four_batches(cfg, B)
    N = batches[0][1].shape[1]
    eps, _ = _draws(e, K, 4 * B, N, seed=7)
    got = e.change_maps(*batches, multiple=1.5, eps=eps, n_draws=K)
    e0 = torch.cat([b[0] for b in batches]); e1 = torch.cat([b[1] for b in batches]); ex = torch.cat([b[2] for b in batches])
    lp = e.log_prob_iw(e1, e.embed(e0), ex, n_draws=K, eps=eps)
    for i, nm in enumerate(("1_0", "0_0", "0_1", "1_1")):
        assert torch.equal(got["log_prob_" + nm], lp[i * B:(i + 1) * B])
        assert torch.equal(got["loss_" + nm], -lp[i * B:(i + 1) * B].mean())
    assert torch.equal(got["change_1_0"], eng.log_prob_to_change(lp[:B], lp[B:2 * B], 1.5))
    assert torch.equal(got["change_0_1"], eng.log_prob_to_change(lp[2 * B:3 * B], lp[3 * B:], 1.5))
    # n_draws = 1: exactly today's result
    eps1 = eps[0]
    a, b = e.change_maps(*batches, multiple=1.5, eps=eps1), e.change_maps(*batches, multiple=1.5, eps=eps1, n_draws=1)
    assert all(torch.equal(a[k], b[k]) for k in a)
    e.close()


def test_evaluate_on_batches_with_draws():
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn", "fp32")
    B, K = 2, 3
    pairs = []
    for i in range(2):
        bs = _four_batches(cfg, B)
        pairs.append((bs[0], bs[1]))
    N = pairs[0][0][1].shape[1]
    epss = [_draws(e, K, 2 * B, N, seed=10 + i)[0] for i in range(2)]
    nats, means = e.evaluate_on_batches(pairs, multiple=2.0, eps=epss, n_draws=K)
    want_nats, want_means = 0.0, []
    for i, (b10, b00) in enumerate(pairs):
        lp = e.log_prob_iw(torch.cat([b10[1], b00[1]]), e.embed(torch.cat([b10[0], b00[0]])), n_draws=K, eps=epss[i])
        ch = eng.log_prob_to_change(lp[:B], lp[B:], 2.0)
        want_means.extend((ch > 0).float().mean(dim=-1).tolist())
        want_nats = (want_nats * i + (-lp[:B].mean() * math.log2(math.e) / e.d_in).item()) / (i + 1)
    assert nats == want_nats and means == want_means
    e1s = [x[0] for x in epss]
    assert e.evaluate_on_batches(pairs, multiple=2.0, eps=e1s) == e.evaluate_on_batches(pairs, multiple=2.0, eps=e1s, n_draws=1)
    e.close()


def test_errors():
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn", "fp32")
    x = batch["extract_1"].to(DEV)
    B, N = x.shape[0], x.shape[1]
    for bad in (0, -2, 2.5, True, "4", None):
        with pytest.raises(fclib.FlowCompareError):
            e.log_prob_iw(x, ctx, n_draws=bad)
    with pytest.raises(fclib.FlowCompareError):
        e.log_prob_iw(x, ctx, n_draws=2, draws_per_pass=0)
    eps, _ = _draws(e, 3, B, N, seed=8)
    for bad_eps in (eps[0], eps[:2], eps[:, :, :5], eps[..., :10]):
        with pytest.raises(fclib.FlowCompareError):
            e.log_prob_iw(x, ctx, n_draws=3, eps=bad_eps)
    with pytest.raises(fclib.FlowCompareError):
        e.log_prob_iw(x, ctx, n_draws=3, eps=eps, eps_cif=torch.zeros(3, e.L, B, N, 8, device=DEV))    # no CIF blocks
    batches = _four_batches(cfg, B)
    with pytest.raises(fclib.FlowCompareError):
        e.change_maps(*batches, n_draws=0)
    with pytest.raises(fclib.FlowCompareError):
        e.evaluate_on_batches([(batches[0], batches[1])], n_draws=1.0)
    # the C entry: too small a workspace, a pass over the row cap
    h, lib = e._flow["handle"], e.lib
    K = 3
    nbytes = lib.fc_flow_log_prob_draws_workspace_bytes(h, B, N, ctx.shape[1], K)
    assert nbytes > lib.fc_flow_workspace_bytes(h, B, N, ctx.shape[1])
    out = torch.empty(K, B, N, device=DEV)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=DEV)
    base = (ws.data_ptr() + 255) // 256 * 256
    s = torch.cuda.current_stream().cuda_stream
    xc = x[..., :6].contiguous()
    rc = lib.fc_flow_log_prob_draws(h, xc.data_ptr(), ctx.data_ptr(), None, eps.data_ptr(), None, K, out.data_ptr(), B, N,
                                    ctx.shape[1], base, nbytes - 256, 0, s)
    assert rc == -4      # FC_ERR_WORKSPACE
    big = (1 << 20) // (B * N) + 1
    assert lib.fc_flow_log_prob_draws_workspace_bytes(h, B, N, ctx.shape[1], big) == -1
    rc = lib.fc_flow_log_prob_draws(h, xc.data_ptr(), ctx.data_ptr(), None, eps.data_ptr(), None, big, out.data_ptr(), B, N,
                                    ctx.shape[1], base, nbytes, 0, s)
    assert rc == -1      # FC_ERR_INVALID_ARG: over 2^20 rows in one pass
    rc = lib.fc_flow_log_prob_draws(h, xc.data_ptr(), ctx.data_ptr(), None, eps.data_ptr(), None, K, out.data_ptr(), B, N,
                                    ctx.shape[1], base, nbytes, 0, s)
    assert rc == 0
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("label", ["dgcnn_attn", "dgcnn_attn_extra", "dgcnn_global"])
def test_points_are_scored_independently(label, precision):
    """log_prob(x[:, :n]) == log_prob(x)[:, :n] bitwise with the same eps prefix, n not a multiple of 128: a point's score
    does not depend on how many points its cloud has."""
    cfg = configs.get_config(label, n_flow_layers=3, sample_size=300, n_samples_context=128)
    fsd, esd = spec.random_state_dicts(cfg, seed=71)
    b = spec.synthetic_batch(cfg, 2, seed=72)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    ctx = e.embed(b["extract_0"].to(DEV))
    x, eps = b["extract_1"].to(DEV), b["eps"].to(DEV)
    extra = None if b["extra_context"] is None else b["extra_context"].to(DEV)
    full = e.log_prob(x, ctx, extra, eps=eps)
    for n in (1, 77, 129, 200, 299):
        part = e.log_prob(x[:, :n], ctx, extra, eps=eps[:, :n])
        assert torch.equal(part, full[:, :n]), (n, (part - full[:, :n]).abs().max().item())
    e.close()
