"""GPU tests of the flow entry points' noise checks: a wrong-shaped `eps` or `eps_cif` raises FlowCompareError naming the
method and the expected shape, before any kernel reads it.  The wrong shapes are oversized, one column too many."""
import re

import pytest
import torch

from flowcompare_b200 import engine as eng, lib as fclib
from oracle.make_golden import fixture_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _setup(name):
    cfg, fsd, esd, batch = fixture_inputs(name)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp32")
    ctx = e.embed(batch["extract_0"].to(DEV))
    return e, ctx, batch["extract_1"].to(DEV), batch


def _raises(what, name, shape):
    return pytest.raises(fclib.FlowCompareError, match=re.escape(f"{what}: {name} must be {list(shape)}"))


def test_wrong_eps_raises():
    e, ctx, x, batch = _setup("tiny_dgcnn_attn")
    B, N = x.shape[:2]
    S = e.D - e.d_in
    bad = torch.zeros(B, N, S + 1, device=DEV)
    calls = {"log_prob": lambda: e.log_prob(x, ctx, eps=bad),
             "forward": lambda: e.forward(x, ctx, eps=bad),
             "attention_maps": lambda: e.attention_maps(x, ctx, eps=bad),
             "log_prob_grad": lambda: e.log_prob_grad(x, ctx, eps=bad)}
    for what, call in calls.items():
        with _raises(what, "eps", (B, N, S)):
            call()
    e.close()


def test_wrong_eps_cif_raises():
    e, ctx, x, batch = _setup("a18_cif")
    B, N = x.shape[:2]
    eps = batch["eps"].to(DEV)
    bad = torch.zeros(e.L, B, N, e.cif_S + 1, device=DEV)
    calls = {"log_prob": lambda: e.log_prob(x, ctx, eps=eps, eps_cif=bad),
             "attention_maps": lambda: e.attention_maps(x, ctx, eps=eps, eps_cif=bad),
             "sample": lambda: e.sample(N, ctx, eps_cif=bad)}
    for what, call in calls.items():
        with _raises(what, "eps_cif", (e.L, B, N, e.cif_S)):
            call()
    e.close()
