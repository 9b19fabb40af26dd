"""GPU tests of the input gradients (engine.log_prob_grad -> fc_flow_log_prob_grad, and autograd on the drop-in adapter): the
gradient matches the fp64 port's autograd gradient, the returned log_prob is bitwise `log_prob`, the result does not depend on
the run, the batch, the pass split or the cloud's other points (also at the 2^16-row pass cap), and the error paths raise."""
import pytest
import torch

from flowcompare_b200 import engine as eng, lib as fclib
from oracle.make_golden import fixture_inputs
from tests.grad_ref import grad_error, port_log_prob_grad

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECISIONS = ["fp32", "tf32x3", "fp16x3"]
ACCURACY = ["tiny_dgcnn_attn", "mid_dgcnn_attn", "tiny_dgcnn_global", "full_dgcnn_global", "tiny_dgcnn_attn_extra",
            "tiny_paconv_attn", "tiny_paconv_attn_extra", "full_dgcnn_attn", "a18_permute_relu", "a18_fullcombiner_noactnorm",
            "a18_expcombiner_global", "a18_identity_augmenter"]
FULL_POINTS = 64       # points scored at full depth (the fp64 port's autograd is the slow part)
_port_cache = {}


def _setup(name, precision="fp32"):
    cfg, fsd, esd, batch = fixture_inputs(name)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    with torch.no_grad():
        ctx = e.embed(batch["extract_0"].to(DEV))
    extra = batch["extra_context"]
    return cfg, fsd, batch, e, ctx, None if extra is None else extra.to(DEV)


def _points(name, batch):
    x, eps = batch["extract_1"], batch["eps"]
    if name.startswith("full_"):
        x, eps = x[:, :FULL_POINTS], eps[:, :FULL_POINTS]
    return x.to(DEV), eps.to(DEV)


def _reference(name):
    """(embedding, fp64 port gradient) of a fixture, once: the embedding of the fp32 path, shared by the three precisions."""
    if name not in _port_cache:
        cfg, fsd, batch, e, ctx, extra = _setup(name, "fp32")
        x, eps = _points(name, batch)
        _port_cache[name] = (ctx, port_log_prob_grad(cfg, fsd, x, ctx, extra, eps)[1])
        e.close()
    return _port_cache[name]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ACCURACY)
def test_gradient_matches_fp64_port(name, precision):
    ctx, g64 = _reference(name)
    cfg, fsd, batch, e, _, extra = _setup(name, precision)
    x, eps = _points(name, batch)
    lp, g = e.log_prob_grad(x, ctx, extra, eps=eps)
    assert g.shape == (x.shape[0], x.shape[1], e.d_in) and torch.isfinite(g).all()
    err = grad_error(g, g64)
    print(f"{name} {precision}: per-point grad error max {err.max().item():.3e} median {err.median().item():.3e} "
          f"(max |g64| {g64.abs().max().item():.3f})")
    assert err.max().item() <= 1e-3 and err.median().item() <= 1e-4
    with torch.no_grad():
        assert torch.equal(lp, e.log_prob(x, ctx, extra, eps=eps))
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_invariant_run_to_run_batch_split_and_prefix(precision):
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn_extra", precision)
    x, eps = _points("tiny_dgcnn_attn_extra", batch)
    B, N = x.shape[0], x.shape[1]
    lp, g = e.log_prob_grad(x, ctx, extra, eps=eps)
    for _ in range(2):
        lp2, g2 = e.log_prob_grad(x, ctx, extra, eps=eps)
        assert torch.equal(lp, lp2) and torch.equal(g, g2)
    lp1, g1 = e.log_prob_grad(x[1:2], ctx[1:2], extra[1:2], eps=eps[1:2])             # one cloud alone vs inside the batch
    assert torch.equal(lp1[0], lp[1]) and torch.equal(g1[0], g[1])
    budget = e.lib.fc_flow_log_prob_grad_workspace_bytes(e._flow["handle"], 1, N, ctx.shape[1])
    lp3, g3 = e.log_prob_grad(x, ctx, extra, eps=eps, workspace_budget=budget)    # one cloud per pass
    assert torch.equal(lp3, lp) and torch.equal(g3, g)
    for n in (1, 77, 93):                                                          # x[:, :n] against x[:, :n] of the whole
        lpn, gn = e.log_prob_grad(x[:, :n], ctx, extra, eps=eps[:, :n])
        assert torch.equal(gn, g[:, :n]) and torch.equal(lpn, lp[:, :n]), n
    e.close()


def test_one_pass_at_the_row_cap():
    """B = 64 clouds of N = 1024 points in one pass (2^16 rows; the checkpoints hold over 2^31 floats at full depth) equals the
    same clouds in passes of 8."""
    cfg, fsd, esd, _ = fixture_inputs("full_dgcnn_attn")
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    B, N, Nc = 64, 1024, 1250
    assert B * N == eng.GRAD_MAX_PASS_ROWS and (e.L + 1) * B * N * e.D > 1 << 31
    gen = torch.Generator(device=DEV).manual_seed(7)
    x = torch.rand(B, N, e.d_in, device=DEV, generator=gen) * 2 - 1
    ctx = torch.randn(B, Nc, e.E, device=DEV, generator=gen)
    eps = torch.randn(B, N, e.D - e.d_in, device=DEV, generator=gen)
    lp, g = e.log_prob_grad(x, ctx, eps=eps)
    budget = e.lib.fc_flow_log_prob_grad_workspace_bytes(e._flow["handle"], 8, N, Nc)
    lp8, g8 = e.log_prob_grad(x, ctx, eps=eps, workspace_budget=budget)
    assert torch.equal(lp, lp8) and torch.equal(g, g8)
    assert torch.isfinite(g).all()
    with torch.no_grad():
        assert torch.equal(lp[:4], e.log_prob(x[:4], ctx[:4], eps=eps[:4]))
    e.close()


@pytest.mark.parametrize("precision", ["fp32", "fp16x3"])
def test_autograd_on_the_adapter(precision):
    cfg, fsd, esd, batch = fixture_inputs("tiny_dgcnn_attn_extra")
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    adapter = eng._FlowAdapter(e)
    x = batch["extract_1"].to(DEV)
    x = torch.cat((x, torch.rand(x.shape[:2] + (2,), device=DEV)), dim=-1)     # columns past input_dim get a zero gradient
    with torch.no_grad():
        ctx = e.embed(batch["extract_0"].to(DEV))
    extra = batch["extra_context"].to(DEV)
    eps = batch["eps"].to(DEV)
    adapter.eps = eps
    with torch.enable_grad():          # other modules of the suite may have switched grad mode off
        plain = adapter.log_prob(x, context=ctx, extra_context=extra)
        assert plain.grad_fn is None
        xg = x.clone().requires_grad_(True)
        lp = adapter.log_prob(xg, context=ctx, extra_context=extra)
        assert lp.grad_fn is not None and torch.equal(lp.detach(), plain)
        w = torch.randn(lp.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
        (gx,) = torch.autograd.grad((w * lp).sum(), xg)
        _, g = e.log_prob_grad(x, ctx, extra, eps=eps)
        assert gx.shape == x.shape
        assert torch.equal(gx[..., :e.d_in], w[..., None] * g) and not gx[..., e.d_in:].any()
        # without injected noise the forward draws eps once, and backward differentiates that same draw
        adapter.eps = None
        torch.manual_seed(11)
        lp = adapter.log_prob(xg, context=ctx, extra_context=extra)
        lp.sum().backward()
        assert xg.grad is not None and torch.isfinite(xg.grad).all()
    # grad mode off: today's path
    with torch.no_grad():
        assert adapter.log_prob(xg, context=ctx, extra_context=extra).grad_fn is None
    e.close()


@pytest.mark.parametrize("name,what", [("a18_spline", "RationalQuadraticSplineCoupling"), ("a18_expo", "ExponentialCoupling"),
                                       ("a18_cif", "CIFblock")])
def test_unsupported_flows_raise(name, what):
    cfg, fsd, batch, e, ctx, extra = _setup(name)
    x = batch["extract_1"].to(DEV)
    with pytest.raises(fclib.FlowCompareError, match=what):
        e.log_prob_grad(x, ctx, extra, eps=batch["eps"].to(DEV))
    adapter = eng._FlowAdapter(e)
    with torch.enable_grad():
        lp = adapter.log_prob(x.clone().requires_grad_(True), context=ctx, extra_context=extra)
        with pytest.raises(fclib.FlowCompareError, match=what):
            lp.sum().backward()
    # the C entry: FC_ERR_UNSUPPORTED before any launch
    B, N = x.shape[0], x.shape[1]
    xc, out = x[..., :e.d_in].contiguous(), torch.empty(B, N, e.d_in, device=DEV)
    rc = e.lib.fc_flow_log_prob_grad(e._flow["handle"], xc.data_ptr(), ctx.data_ptr(), None, out.data_ptr(), out.data_ptr(),
                                     out.data_ptr(), B, N, ctx.shape[1], out.data_ptr(), 0, 0, torch.cuda.current_stream().cuda_stream)
    assert rc == -5
    e.close()


def test_errors():
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn")
    x, eps = _points("tiny_dgcnn_attn", batch)
    B, N = x.shape[0], x.shape[1]
    for bad in (eps[0], eps[:, :5], eps[..., :10], torch.zeros(B, N, e.D, device=DEV)):
        with pytest.raises(fclib.FlowCompareError):
            e.log_prob_grad(x, ctx, eps=bad)
    adapter = eng._FlowAdapter(e)
    adapter.eps = eps
    with torch.enable_grad():
        xg = x.clone().requires_grad_(True)
        lp = adapter.log_prob(xg, context=ctx.clone().requires_grad_(True))
        with pytest.raises(fclib.FlowCompareError, match="context"):
            lp.sum().backward()
    # the C entry: no transposed weights attached, too small a workspace, a pass over the row cap
    e2 = eng.FlowCompareB200((fsd, fixture_inputs("tiny_dgcnn_attn")[2]), cfg, device=DEV)
    h2, lib = e2._flow["handle"], e2.lib
    nbytes = lib.fc_flow_log_prob_grad_workspace_bytes(h2, B, N, ctx.shape[1])
    assert nbytes > lib.fc_flow_workspace_bytes(h2, B, N, ctx.shape[1])
    assert lib.fc_flow_log_prob_grad_workspace_bytes(h2, (1 << 16) // N + 1, N, ctx.shape[1]) == -1
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=DEV)
    base = (ws.data_ptr() + 255) // 256 * 256
    s = torch.cuda.current_stream().cuda_stream
    lp_out, g_out = torch.empty(B, N, device=DEV), torch.empty(B, N, e.d_in, device=DEV)
    xc = x[..., :e.d_in].contiguous()
    args = lambda nb: (h2, xc.data_ptr(), ctx.data_ptr(), None, eps.data_ptr(), lp_out.data_ptr(), g_out.data_ptr(), B, N,
                       ctx.shape[1], base, nb, 0, s)
    assert lib.fc_flow_log_prob_grad(*args(nbytes)) == -6          # FC_ERR_MODEL: fc_flow_set_grad not called
    e2._ensure_grad()
    assert lib.fc_flow_log_prob_grad(*args(nbytes - 256)) == -4    # FC_ERR_WORKSPACE
    assert lib.fc_flow_log_prob_grad(*args(nbytes)) == 0
    with torch.no_grad():
        assert torch.equal(lp_out, e2.log_prob(x, ctx, eps=eps))
    e2.close()
    e.close()
