"""GPU tests of the attention score gradients (engine.attention_score_grads -> fc_flow_attention_score_grads ->
attention_score_grad_kernel): d lp_i / d s_ij of every attention block against the fp64 port's retained `sim.grad`, log_prob and
grad bitwise `log_prob_grad`'s, the result independent of the run, the batch, the pass split and the query list, the layer sum,
the kernel's own contract (fp64 closed form, tails, zero row sums, NaN rows, 64-bit offsets) and the error paths."""
import numpy as np
import pytest
import torch

from flowcompare_b200 import configs, engine as eng, lib as fclib, spec
from oracle.make_golden import fixture_inputs
from tests.attention_score_grads_ref import port_score_grads, row_error, score_grads

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PRECISIONS = ["fp32", "tf32x3", "fp16x3"]
# the attention fixtures of tests/test_log_prob_grad_gpu.py (the global ones have no attention over context points)
ACCURACY = ["tiny_dgcnn_attn", "mid_dgcnn_attn", "full_dgcnn_attn", "tiny_dgcnn_attn_extra", "tiny_paconv_attn",
            "tiny_paconv_attn_extra", "a18_permute_relu", "a18_fullcombiner_noactnorm", "a18_identity_augmenter"]
FULL_POINTS = 64       # points scored at full depth (the fp64 port's backward is the slow part)
# (worst row, median row) bounds.  The value is P_ij (dO_i.v_j - dO_i.o_i): a difference of two dot products, each rounded to fp32
# at the scale of |dO_i| |v_j|.  The seeded PAConv embedders give nearly the same embedding to every context point, so there
# |v_j - o_i| is ~0.2 % of |v_j| (~1.5 % for DGCNN) and that rounding is ~7x larger relative to the value: the closed form
# evaluated in fp32 on the fp64 port's own q, k, v, o and dO reaches 8.7e-4 worst / 9.6e-5 median on tiny_paconv_attn.  The
# kernel alone is within 2e-5 of fp64 (test_kernel_against_fp64).
BOUNDS = {"tiny_paconv_attn": (3e-3, 3e-4), "tiny_paconv_attn_extra": (3e-3, 3e-4)}
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


def _reference(monkeypatch, name):
    """(embedding, {block: fp64 d lp_i / d s_ij}) of a fixture, once: the embedding of the fp32 path, shared by the precisions."""
    if name not in _port_cache:
        cfg, fsd, batch, e, ctx, extra = _setup(name, "fp32")
        x, eps = _points(name, batch)
        _, rec = port_score_grads(monkeypatch, cfg, fsd, x, ctx, extra, eps)
        _port_cache[name] = (ctx, {p: g.detach() for p, g in score_grads(rec).items()})
        e.close()
    return _port_cache[name]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ACCURACY)
def test_score_grads_match_fp64_port(monkeypatch, name, precision):
    """Per query row, max_j |got - fp64| over max_j |fp64| (the values are of order P_ij, so each row is judged at its own scale;
    the normaliser is floored at 1e-6 of the block's largest value, for rows whose gradient is within fp32 noise of zero), against
    the input-gradient tests' bounds, 1e-3 worst and 1e-4 median (BOUNDS: the PAConv fixtures).  Also: log_prob and grad are
    bitwise log_prob_grad's."""
    ctx, want = _reference(monkeypatch, name)
    cfg, fsd, batch, e, _, extra = _setup(name, precision)
    x, eps = _points(name, batch)
    lp, g, maps = e.attention_score_grads(x, ctx, extra, eps=eps)
    assert list(maps) == e.attention_layer_names == list(want)
    B, N, Nc = x.shape[0], x.shape[1], ctx.shape[1]
    err = torch.cat([row_error(maps[n], want[n]) for n in maps])
    for m in maps.values():
        assert m.shape == (B, N, Nc) and torch.isfinite(m).all()
    print(f"{name} {precision}: {len(maps)} blocks, per-row error max {err.max().item():.3e} median {err.median().item():.3e} "
          f"(max |fp64| {max(w.abs().max().item() for w in want.values()):.3e})")
    worst, median = BOUNDS.get(name, (1e-3, 1e-4))
    assert err.max().item() <= worst and err.median().item() <= median
    lp2, g2 = e.log_prob_grad(x, ctx, extra, eps=eps)
    assert torch.equal(lp, lp2) and torch.equal(g, g2)
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_query_subset_rows_equal_full_maps(precision):
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn", precision)
    x, eps = _points("tiny_dgcnn_attn", batch)
    lp, g, full = e.attention_score_grads(x, ctx, eps=eps)
    q = [95, 3, 17, 3, 0, 64, 95, 40]                  # unsorted, with repeats, in both 64-row halves of a CTA
    lp_s, g_s, sub = e.attention_score_grads(x, ctx, eps=eps, queries=q)
    name = e.attention_layer_names[2]
    _, _, sub_t = e.attention_score_grads(x, ctx, eps=eps, queries=torch.tensor(q, device=DEV), layers=[name])
    assert torch.equal(lp_s, lp) and torch.equal(g_s, g)
    for n in full:
        assert sub[n].shape == (x.shape[0], len(q), ctx.shape[1])
        assert torch.equal(sub[n], full[n][:, q])
    assert list(sub_t) == [name] and torch.equal(sub_t[name], full[name][:, q])
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_invariant_run_to_run_batch_and_split(precision):
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn_extra", precision)
    x, eps = _points("tiny_dgcnn_attn_extra", batch)
    N, Nc = x.shape[1], ctx.shape[1]
    lp, g, m = e.attention_score_grads(x, ctx, extra, eps=eps)
    _, _, ms = e.attention_score_grads(x, ctx, extra, eps=eps, sum_layers=True)
    lp2, g2, m2 = e.attention_score_grads(x, ctx, extra, eps=eps)
    assert torch.equal(lp, lp2) and torch.equal(g, g2) and all(torch.equal(m[n], m2[n]) for n in m)
    lp1, g1, m1 = e.attention_score_grads(x[1:2], ctx[1:2], extra[1:2], eps=eps[1:2])      # one cloud alone vs inside the batch
    assert torch.equal(lp1[0], lp[1]) and torch.equal(g1[0], g[1]) and all(torch.equal(m1[n][0], m[n][1]) for n in m)
    budget = e.lib.fc_flow_log_prob_grad_workspace_bytes(e._flow["handle"], 1, N, Nc)   # one cloud per pass
    lp3, g3, m3 = e.attention_score_grads(x, ctx, extra, eps=eps, workspace_budget=budget)
    assert torch.equal(lp3, lp) and torch.equal(g3, g) and all(torch.equal(m3[n], m[n]) for n in m)
    _, _, ms3 = e.attention_score_grads(x, ctx, extra, eps=eps, workspace_budget=budget, sum_layers=True)
    assert torch.equal(ms3, ms)
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_sum_layers_is_the_walk_order_fp32_sum(precision):
    """sum_layers adds the blocks in the backward walk's order: the last coupling layer's first, the augmenter's last."""
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn", precision)
    x, eps = _points("tiny_dgcnn_attn", batch)
    names = e.attention_layer_names
    q = [7, 90, 7, 33]
    for layers, queries in ((None, None), ([names[3], names[0], names[1]], q), ([names[2]], None)):
        lp, g, per = e.attention_score_grads(x, ctx, eps=eps, layers=layers, queries=queries)
        lp_s, g_s, tot = e.attention_score_grads(x, ctx, eps=eps, layers=layers, queries=queries, sum_layers=True)
        want = torch.zeros_like(tot)
        for n in reversed(names):
            if n in per:
                want = want + per[n]
        assert torch.equal(tot, want), layers
        assert torch.equal(lp_s, lp) and torch.equal(g_s, g)
    e.close()


def test_many_slots_past_2e31_elements():
    """A 3-layer model (4 blocks) at B = 16 clouds of 1024 points against 33000 context points: 2.16e9 values in one allocation,
    the last block crossing 2^31.  The first and last block equal single-block calls bitwise, so no offset wraps."""
    cfg = configs.get_config("dgcnn_attn", n_flow_layers=3)
    fsd, esd = spec.random_state_dicts(cfg, seed=5)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    B, N, Nc = 16, 1024, 33000
    gen = torch.Generator(device=DEV).manual_seed(9)
    x = torch.rand(B, N, e.d_in, device=DEV, generator=gen) * 2 - 1
    ctx = torch.randn(B, Nc, e.E, device=DEV, generator=gen)
    eps = torch.randn(B, N, e.D - e.d_in, device=DEV, generator=gen)
    names = e.attention_layer_names
    _, _, allm = e.attention_score_grads(x, ctx, eps=eps)
    assert len(allm) == 4 and 4 * B * N * Nc > 2 ** 31
    for name in (names[0], names[3]):
        _, _, one = e.attention_score_grads(x, ctx, eps=eps, layers=[name])
        assert torch.equal(allm[name], one[name]), name
        del one
    del allm
    e.close()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ the kernel alone
def _op_inputs(B, N, Nc, seed):
    """Random q, k | v, dO (fp32) and o = softmax(q k^T / 8) v formed in fp64 from them, rounded once to fp32."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, N, 64, generator=g)
    kv = torch.randn(B, Nc, 128, generator=g)
    dO = torch.randn(B, N, 64, generator=g)
    P = torch.softmax(q.double() @ kv[..., :64].double().transpose(1, 2) * 0.125, dim=-1)
    o = (P @ kv[..., 64:].double()).float()
    return q, kv, o, dO


def _op_fp64(q, kv, o, dO):
    P = torch.softmax(q.double() @ kv[..., :64].double().transpose(1, 2) * 0.125, dim=-1)
    dp = dO.double() @ kv[..., 64:].double().transpose(1, 2)
    D = (dO.double() * o.double()).sum(-1, keepdim=True)
    return P * (dp - D)


def _op_call(q, kv, o, dO, out, qidx=None, accumulate=0):
    B, N, Nc = q.shape[0], q.shape[1], kv.shape[1]
    n_query = N if qidx is None else qidx.numel()
    lib = fclib.load()
    return lib.fc_attention_score_grad(q.data_ptr(), 64, kv.data_ptr(), 128, o.data_ptr(), 64, dO.data_ptr(), 64,
                                       0 if qidx is None else qidx.data_ptr(), n_query, out.data_ptr(), accumulate, B, N, Nc,
                                       0.125, torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("B,N,Nc", [(2, 70, 130), (3, 129, 6), (1, 200, 1), (2, 256, 1251), (1, 300, 64)])
def test_kernel_against_fp64(B, N, Nc):
    """Query tails past 128-row tiles, key counts that are not multiples of 64 or of 4 (scalar stores), one key (P = 1, every
    value 0 up to rounding); accumulate mode is one rounded add; query lists pick rows; clouds do not see each other."""
    q, kv, o, dO = _op_inputs(B, N, Nc, seed=B * 1000 + N + Nc)
    want = _op_fp64(q, kv, o, dO)
    qd, kvd, od, dOd = (t.to(DEV) for t in (q, kv, o, dO))
    out = torch.empty(B, N, Nc, device=DEV)
    assert _op_call(qd, kvd, od, dOd, out) == 0
    got = out.cpu().double()
    if Nc == 1:         # o = v exactly, and dO.v, dO.o are the same fma chain
        assert not got.any()
    else:
        err = row_error(out, want).max().item()
        rsum = (got.sum(-1).abs() / got.abs().sum(-1)).max().item()
        print(f"B={B} N={N} Nc={Nc}: per-row error {err:.3e}, max |row sum| / sum |row| {rsum:.3e}")
        assert err <= 2e-5
        assert rsum <= 1e-4
    base = torch.randn(B, N, Nc, device=DEV)
    acc = base.clone()
    assert _op_call(qd, kvd, od, dOd, acc, accumulate=1) == 0
    assert torch.equal(acc, base + out)
    idx = torch.tensor([N - 1, 0, N // 2, N - 1], dtype=torch.int32, device=DEV)
    sub = torch.empty(B, 4, Nc, device=DEV)
    assert _op_call(qd, kvd, od, dOd, sub, qidx=idx) == 0
    assert torch.equal(sub, out[:, idx.long()])
    one = torch.empty(1, N, Nc, device=DEV)
    assert _op_call(qd[B - 1:], kvd[B - 1:], od[B - 1:], dOd[B - 1:], one) == 0
    assert torch.equal(one[0], out[B - 1])


def test_kernel_nan_gives_nan_rows():
    """A NaN in q or dO poisons its own row only; a NaN in one key poisons every row of its cloud."""
    B, N, Nc = 2, 70, 130
    q, kv, o, dO = _op_inputs(B, N, Nc, seed=5)
    q[0, 5, 7] = float("nan")
    dO[0, 9, 1] = float("nan")
    kv[1, 9, 3] = float("nan")              # cloud 1, key 9
    out = torch.empty(B, N, Nc, device=DEV)
    assert _op_call(q.to(DEV), kv.to(DEV), o.to(DEV), dO.to(DEV), out) == 0
    out = out.cpu()
    assert torch.isnan(out[0, 5]).all() and torch.isnan(out[0, 9]).all()
    rows = [r for r in range(N) if r not in (5, 9)]
    assert torch.isfinite(out[0, rows]).all()
    assert torch.isnan(out[1]).all()
    want = _op_fp64(q[:1], kv[:1], o[:1], dO[:1])[0]
    assert row_error(out[0, rows], want[rows]).max().item() <= 2e-5


def test_kernel_offsets_past_2e31_elements():
    """3 clouds x 1024 queries x 720000 keys = 2.2e9 values (8.8 GB): the last cloud's rows equal a one-cloud call, and
    accumulating the output onto itself doubles it exactly there."""
    B, N, Nc = 3, 1024, 720000
    assert B * N * Nc > 2 ** 31
    gen = torch.Generator(device=DEV).manual_seed(3)
    q = torch.randn(B, N, 64, device=DEV, generator=gen)
    kv = torch.randn(B, Nc, 128, device=DEV, generator=gen)
    dO = torch.randn(B, N, 64, device=DEV, generator=gen)
    o = torch.randn(B, N, 64, device=DEV, generator=gen)
    out = torch.empty(B, N, Nc, device=DEV)
    assert _op_call(q, kv, o, dO, out) == 0
    idx = torch.tensor([N - 1, 0], dtype=torch.int32, device=DEV)
    one = torch.empty(1, 2, Nc, device=DEV)
    assert _op_call(q[2:], kv[2:], o[2:], dO[2:], one, qidx=idx) == 0
    assert torch.equal(one[0, 0], out[2, N - 1]) and torch.equal(one[0, 1], out[2, 0])
    last = out[2, N - 1].clone()
    assert torch.isfinite(last).all()
    assert _op_call(q, kv, o, dO, out, accumulate=1) == 0
    assert torch.equal(out[2, N - 1], 2 * last)
    del out, one, kv
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ errors
def _raw_call(e, x, ctx, eps, slots, n_query=None, nbytes=None):
    B, N, Nc = x.shape[0], x.shape[1], ctx.shape[1]
    n_query = N if n_query is None else n_query
    xc = x[..., :e.d_in].contiguous()
    maps = torch.empty(max(1, len(slots)), B, n_query, Nc, device=DEV)
    lp, g = torch.empty(B, N, device=DEV), torch.empty(B, N, e.d_in, device=DEV)
    need = e.lib.fc_flow_log_prob_grad_workspace_bytes(e._flow["handle"], B, N, Nc)
    ws = torch.empty(max(need, 0) + 256, dtype=torch.uint8, device=DEV)
    base = (ws.data_ptr() + 255) // 256 * 256
    s = np.asarray(slots, dtype=np.int32)
    rc = e.lib.fc_flow_attention_score_grads(e._flow["handle"], xc.data_ptr(), ctx.data_ptr(), None,
                                             eps.data_ptr() if eps.numel() else None, s.ctypes.data, len(slots), None, n_query, 0,
                                             maps.data_ptr(), lp.data_ptr(), g.data_ptr(), B, N, Nc, base,
                                             need if nbytes is None else nbytes(need), 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


def test_errors():
    # global embedding: no attention over context points, in the engine and at the C entry
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_global")
    x, eps = _points("tiny_dgcnn_global", batch)
    with pytest.raises(fclib.FlowCompareError, match="global"):
        e.attention_score_grads(x, ctx, eps=eps)
    assert _raw_call(e, x, ctx.reshape(ctx.shape[0], 1, -1).contiguous(), eps, [1]) == -5      # FC_ERR_UNSUPPORTED
    e.close()
    # a spline flow: the transform is named, as by log_prob_grad
    cfg, fsd, batch, e, ctx, extra = _setup("a18_spline")
    with pytest.raises(fclib.FlowCompareError, match="RationalQuadraticSplineCoupling"):
        e.attention_score_grads(batch["extract_1"].to(DEV), ctx, eps=batch["eps"].to(DEV))
    e.close()
    cfg, fsd, batch, e, ctx, extra = _setup("tiny_dgcnn_attn")
    x, eps = _points("tiny_dgcnn_attn", batch)
    N = x.shape[1]
    assert _raw_call(e, x, ctx, eps, [1]) == -6                    # FC_ERR_MODEL: fc_flow_set_grad not called
    for layers in (["transforms.2.pre_conditioner.attn"], []):                   # transforms.2 is an ActNorm; no layers
        with pytest.raises(fclib.FlowCompareError):
            e.attention_score_grads(x, ctx, eps=eps, layers=layers)
    for bad in ([N], [-1], [0, N + 5], [], [1.0, 2.0]):
        with pytest.raises(fclib.FlowCompareError):
            e.attention_score_grads(x, ctx, eps=eps, queries=bad)
    # the C entry's argument and workspace errors
    e._ensure_grad()
    assert _raw_call(e, x, ctx, eps, [0, 1, 3]) == 0
    assert _raw_call(e, x, ctx, eps, [2, 1]) == -1                 # unsorted
    assert _raw_call(e, x, ctx, eps, [1, 1]) == -1                 # repeated
    assert _raw_call(e, x, ctx, eps, [4]) == -1                    # 3 layers: slots 0..3
    assert _raw_call(e, x, ctx, eps, [1], n_query=N - 1) == -1     # no query list, n_query != N
    assert _raw_call(e, x, ctx, eps, [1], nbytes=lambda need: need - 256) == -4     # FC_ERR_WORKSPACE
    e.close()
    # identity augmenter: no transforms.0.attn, slot 0 is an argument error
    cfg, fsd, batch, e, ctx, extra = _setup("a18_identity_augmenter")
    x, eps = _points("a18_identity_augmenter", batch)
    with pytest.raises(fclib.FlowCompareError):
        e.attention_score_grads(x, ctx, eps=eps, layers=["transforms.0.attn"])
    e._ensure_grad()
    assert _raw_call(e, x, ctx, eps, [0, 1]) == -1
    assert _raw_call(e, x, ctx, eps, [1]) == 0
    e.close()
