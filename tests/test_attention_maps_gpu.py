"""GPU tests of the attention maps (engine.attention_maps -> fc_flow_attention_maps -> attention_maps_kernel): the softmax
weights of every attention block against the oracle port run in float64 on the same fp32 context embedding the engine gets
(so the two sides differ only by the flow), the contract of the kernel (rows sum to 1, deterministic, batch invariant, query
subsets, 64-bit offsets, tails) and that capturing leaves the forward pass bitwise unchanged."""
import numpy as np
import pytest
import torch

from flowcompare_b200 import configs, engine as eng, lib as fclib, spec
from oracle.make_golden import fixture_inputs
from tests.attention_maps_ref import port_attention_maps

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
DEV = "cuda:0"
PRECISIONS = ["fp32", "tf32x3", "fp16x3"]


def _setup(name, precision):
    cfg, fsd, esd, batch = fixture_inputs(name)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    ctx = e.embed(batch["extract_0"].to(DEV))
    return cfg, fsd, batch, e, ctx


def _noise(batch):
    extra = batch["extra_context"]
    return dict(extra_context=None if extra is None else extra.to(DEV), eps=batch["eps"].to(DEV),
                eps_cif=batch["eps_cif"].to(DEV) if "eps_cif" in batch else None)


def _check_maps(maps):
    for m in maps.values():
        m = m.cpu()
        assert torch.isfinite(m).all()
        assert (m >= 0).all() and (m <= 1).all()
        assert (m.double().sum(-1) - 1).abs().max().item() < 1e-5


def _against_port(monkeypatch, cfg, fsd, x, ctx, extra, eps, eps_cif, maps, keep=None):
    """Max |maps - fp64 port| over the blocks in `maps`."""
    _, want = port_attention_maps(monkeypatch, cfg, fsd, x, ctx, extra, eps, eps_cif, keep=keep)
    assert set(maps) <= set(want)
    return max((m.cpu().double() - want[n]).abs().max().item() for n, m in maps.items())


def _fixture_against_port(monkeypatch, name, precision):
    cfg, fsd, batch, e, ctx = _setup(name, precision)
    lp, maps = e.attention_maps(batch["extract_1"].to(DEV), ctx, **_noise(batch))
    assert list(maps) == e.attention_layer_names
    B, N, Nc = ctx.shape[0], batch["extract_1"].shape[1], ctx.shape[1]
    assert all(m.shape == (B, N, Nc) for m in maps.values())
    _check_maps(maps)
    err = _against_port(monkeypatch, cfg, fsd, batch["extract_1"], ctx, batch["extra_context"], batch["eps"],
                        batch.get("eps_cif"), maps)
    print(f"{name} {precision}: {len(maps)} blocks, max |maps - fp64 port| {err:.3e}")
    e.close()
    return err


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "tiny_paconv_attn", "mid_dgcnn_attn"])
def test_maps_match_fp64_port(monkeypatch, name, precision):
    assert _fixture_against_port(monkeypatch, name, precision) <= 2e-5


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["a18_spline", "a18_expo", "a18_cif", "a18_identity_augmenter"])
def test_a18_maps_match_fp64_port(monkeypatch, name, precision):
    """The other couplings, the CIF block's naming (transforms.{t}.flow.pre_conditioner.attn) and an identity augmenter."""
    assert _fixture_against_port(monkeypatch, name, precision) <= 2e-5


def test_full_depth_maps_match_fp64_port(monkeypatch):
    """115 layers, B = 1, 3xFP16: the first and second block, one in the middle and the last.  The latent reaching the late
    layers carries the forward's accumulated drift (<= 1e-3 nats on the log-prob), hence the looser bound."""
    cfg, fsd, batch, e, ctx = _setup("full_dgcnn_attn", "fp16x3")
    names = e.attention_layer_names
    assert len(names) == 116
    pick = [names[0], names[1], names[58], names[115]]
    _, maps = e.attention_maps(batch["extract_1"].to(DEV), ctx, layers=pick, **_noise(batch))
    assert list(maps) == pick
    _check_maps(maps)
    err = _against_port(monkeypatch, cfg, fsd, batch["extract_1"], ctx, None, batch["eps"], None, maps, keep=set(pick))
    print(f"full_dgcnn_attn fp16x3 slots 0, 1, 58, 115: max |maps - fp64 port| {err:.3e}")
    assert err <= 1e-4
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", ["tiny_dgcnn_attn_extra", "a18_cif"])
def test_capture_leaves_log_prob_bitwise_unchanged(name, precision):
    cfg, fsd, batch, e, ctx = _setup(name, precision)
    x = batch["extract_1"].to(DEV)
    lp_maps, _ = e.attention_maps(x, ctx, **_noise(batch))
    lp = e.log_prob(x, ctx, **_noise(batch))
    assert torch.equal(lp_maps, lp)
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_query_subset_rows_equal_full_maps(precision):
    cfg, fsd, batch, e, ctx = _setup("tiny_dgcnn_attn", precision)
    x = batch["extract_1"].to(DEV)
    _, full = e.attention_maps(x, ctx, **_noise(batch))
    q = [95, 3, 17, 3, 0, 64, 95, 40]                  # unsorted, with repeats, in both 64-row halves of a CTA
    _, sub = e.attention_maps(x, ctx, queries=q, **_noise(batch))
    _, sub_t = e.attention_maps(x, ctx, queries=torch.tensor(q, device=DEV), layers=[e.attention_layer_names[2]], **_noise(batch))
    for name in full:
        assert sub[name].shape == (x.shape[0], len(q), ctx.shape[1])
        assert torch.equal(sub[name], full[name][:, q])
    assert torch.equal(sub_t[e.attention_layer_names[2]], full[e.attention_layer_names[2]][:, q])
    e.close()


@pytest.mark.parametrize("precision", PRECISIONS)
def test_maps_batch_invariant_and_deterministic(precision):
    cfg = configs.get_config("dgcnn_attn", n_flow_layers=3, sample_size=200, n_samples_context=300)
    fsd, esd = spec.random_state_dicts(cfg, seed=3)
    batch = spec.synthetic_batch(cfg, 3, seed=4)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    ctx = e.embed(batch["extract_0"].to(DEV))
    x, eps = batch["extract_1"].to(DEV), batch["eps"].to(DEV)
    _, a = e.attention_maps(x, ctx, eps=eps)
    _, a2 = e.attention_maps(x, ctx, eps=eps)
    _, one = e.attention_maps(x[1:2], ctx[1:2], eps=eps[1:2])
    for name in a:
        assert torch.equal(a[name], a2[name])
        assert torch.equal(a[name][1:2], one[name])
    e.close()


def test_many_slots_equal_single_slot_calls_past_2e31_elements():
    """All 116 blocks of the full-depth model at B = 16 (1024 x 1250 weights per cloud and block: 2.38e9 elements, 9.5 GB in
    one allocation): the first, a middle and the last block equal single-block calls bitwise, so no offset wraps at 2^31."""
    cfg = configs.get_config("dgcnn_attn")
    fsd, esd = spec.random_state_dicts(cfg, seed=0)
    B = 16
    batch = spec.synthetic_batch(cfg, B, seed=100)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    ctx = e.embed(batch["extract_0"].to(DEV))
    x, eps = batch["extract_1"].to(DEV), batch["eps"].to(DEV)
    names = e.attention_layer_names
    _, allm = e.attention_maps(x, ctx, eps=eps)
    first = next(iter(allm.values()))
    assert len(allm) * first.numel() > 2 ** 31
    for name in (names[0], names[57], names[115]):
        _, one = e.attention_maps(x, ctx, eps=eps, layers=[name])
        assert torch.equal(allm[name], one[name]), name
        del one
    del allm, first
    e.close()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("B,N,Nc", [(2, 96, 1), (2, 130, 4097), (2, 96, 6)])
def test_edge_shapes_against_port(monkeypatch, precision, B, N, Nc):
    """One context point (every weight exactly 1), a key count with a tail of one past 64-key tiles with a query tail past a
    128-row tile, and a tiny context; random context embeddings are handed to the engine and the port alike."""
    cfg = configs.tiny_config("dgcnn_attn")
    fsd, esd = spec.random_state_dicts(cfg, seed=9)
    batch = spec.synthetic_batch(cfg, B, seed=10, n_target=N)
    g = torch.Generator().manual_seed(Nc)
    ctx = torch.randn(B, Nc, cfg["input_embedding_dim"], generator=g)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision=precision)
    _, maps = e.attention_maps(batch["extract_1"].to(DEV), ctx.to(DEV), eps=batch["eps"].to(DEV))
    _check_maps(maps)
    if Nc == 1:
        assert all(bool((m == 1).all()) for m in maps.values())
    err = _against_port(monkeypatch, cfg, fsd, batch["extract_1"], ctx, None, batch["eps"], None, maps)
    print(f"B={B} N={N} Nc={Nc} {precision}: max |maps - fp64 port| {err:.3e}")
    assert err <= 2e-5
    e.close()


def _raw_call(e, batch, ctx, slots, n_query=None, qidx=None):
    x = batch["extract_1"][..., :e.d_in].contiguous().to(DEV)
    B, N, Nc = x.shape[0], x.shape[1], ctx.shape[1]
    n_query = N if n_query is None else n_query
    eps = batch["eps"].to(DEV).contiguous()
    maps = torch.empty(max(1, len(slots)), B, n_query, Nc, device=DEV)
    lp = torch.empty(B, N, device=DEV)
    nbytes = e.lib.fc_flow_workspace_bytes(e._flow["handle"], B, N, Nc)
    ws = e._workspace(nbytes)
    s = np.asarray(slots, dtype=np.int32)
    rc = e.lib.fc_flow_attention_maps(e._flow["handle"], x.data_ptr(), ctx.data_ptr(), 0, eps.data_ptr() if eps.numel() else 0,
                                      0, s.ctypes.data, len(slots), 0 if qidx is None else qidx.data_ptr(), n_query,
                                      maps.data_ptr(), lp.data_ptr(), B, N, Nc, ws, nbytes, e.precision,
                                      torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


def test_errors():
    # global embedding: no attention over context points, in the engine and at the C entry
    cfg, fsd, batch, e, ctx = _setup("tiny_dgcnn_global", "fp32")
    assert e.attention_layer_names == []
    with pytest.raises(fclib.FlowCompareError):
        e.attention_maps(batch["extract_1"].to(DEV), ctx, eps=batch["eps"].to(DEV))
    assert _raw_call(e, batch, ctx.reshape(ctx.shape[0], 1, -1).contiguous(), [1]) == -5      # FC_ERR_UNSUPPORTED
    e.close()
    cfg, fsd, batch, e, ctx = _setup("tiny_dgcnn_attn", "fp32")
    x, eps = batch["extract_1"].to(DEV), batch["eps"].to(DEV)
    N = x.shape[1]
    with pytest.raises(fclib.FlowCompareError):
        e.attention_maps(x, ctx, eps=eps, layers=["transforms.2.pre_conditioner.attn"])     # transforms.2 is an ActNorm
    for bad in ([N], [-1], [0, N + 5]):
        with pytest.raises(fclib.FlowCompareError):
            e.attention_maps(x, ctx, eps=eps, queries=bad)
    assert _raw_call(e, batch, ctx, [0, 1, 3]) == 0
    assert _raw_call(e, batch, ctx, [2, 1]) == -1                 # unsorted
    assert _raw_call(e, batch, ctx, [1, 1]) == -1                 # repeated
    assert _raw_call(e, batch, ctx, [4]) == -1                    # 3 layers: slots 0..3
    assert _raw_call(e, batch, ctx, [1], n_query=N - 1) == -1     # no query list, n_query != N
    e.close()
    # identity augmenter: no transforms.0.attn, slot 0 is an argument error
    cfg, fsd, batch, e, ctx = _setup("a18_identity_augmenter", "fp32")
    assert "transforms.0.attn" not in e.attention_layer_names
    with pytest.raises(fclib.FlowCompareError):
        e.attention_maps(batch["extract_1"].to(DEV), ctx, layers=["transforms.0.attn"], eps=batch["eps"].to(DEV))
    assert _raw_call(e, batch, ctx, [0, 1]) == -1
    assert _raw_call(e, batch, ctx, [1]) == 0
    e.close()


def test_nan_gives_nan_rows():
    """A NaN in q poisons its own row only; a NaN in one key poisons every row of its cloud (never a silently renormalised row)."""
    lib = fclib.load()
    B, N, Nc = 2, 70, 130
    g = torch.Generator().manual_seed(5)
    q = torch.randn(B * N, 64, generator=g)
    kv = torch.randn(B * Nc, 128, generator=g)
    q[5, 7] = float("nan")
    kv[Nc + 9, 3] = float("nan")            # cloud 1, key 9
    qd, kvd = q.to(DEV), kv.to(DEV)
    out = torch.empty(B, N, Nc, device=DEV)
    assert lib.fc_attention_maps(qd.data_ptr(), 64, kvd.data_ptr(), 128, 0, N, out.data_ptr(), B, N, Nc, 0.125,
                                 torch.cuda.current_stream().cuda_stream) == 0
    out = out.cpu()
    assert torch.isnan(out[0, 5]).all()
    assert torch.isfinite(out[0, :5]).all() and torch.isfinite(out[0, 6:]).all()
    assert torch.isnan(out[1]).all()
    want = torch.softmax((q[:N].double() @ kv[:Nc, :64].double().t()) * 0.125, dim=-1)
    rows = [r for r in range(N) if r != 5]
    assert (out[0, rows].double() - want[rows]).abs().max().item() < 2e-6
