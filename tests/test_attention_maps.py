"""CPU side of the attention maps (engine.attention_maps, fc_flow_attention_maps): the packing's list of attention-block names
against the reference's module names, and the port recorder the GPU tests compare against (tests/attention_maps_ref.py)."""
import re

import pytest
import torch

from flowcompare_b200 import configs, packing, spec
from oracle import port
from oracle.make_golden import FIXTURES, fixture_inputs
from tests.attention_maps_ref import port_attention_maps

torch.set_grad_enabled(False)


def _to_q_prefixes(cfg):
    """Prefixes of every `*.attn.fn.attention.to_q.weight` of the flow's state_dict, in transform order."""
    suffix = ".fn.attention.to_q.weight"
    pre = [k[:-len(suffix)] for k in spec.flow_param_shapes(cfg) if k.endswith(suffix)]
    return sorted(pre, key=lambda p: int(re.match(r"transforms\.(\d+)\.", p).group(1)))


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_block_names_are_the_state_dict_attention_prefixes(name):
    label, over, *_ = FIXTURES[name]
    cfg = configs.get_config(label, **over)
    names = packing.attention_block_names(cfg)
    if configs.derive(cfg)["global"]:
        assert names == []          # the global embedder's conditioners have no attention over context points
        return
    assert names == _to_q_prefixes(cfg)
    assert len(names) == cfg["n_flow_layers"] + (1 if cfg["latent_dim"] > cfg["input_dim"] else 0)


def test_block_names_cover_cif_and_identity_augmenter():
    cif = FIXTURES["a18_cif"]
    names = packing.attention_block_names(configs.get_config(cif[0], **cif[1]))
    assert names[0] == "transforms.0.attn" and names[1] == "transforms.1.flow.pre_conditioner.attn"
    ident = FIXTURES["a18_identity_augmenter"]
    names = packing.attention_block_names(configs.get_config(ident[0], **ident[1]))
    assert "transforms.0.attn" not in names and names[0] == "transforms.1.pre_conditioner.attn"


@pytest.mark.parametrize("name", ["tiny_dgcnn_attn", "tiny_dgcnn_attn_extra", "a18_cif"])
def test_recorder_restates_the_port(monkeypatch, name):
    """The recorder's weights times v (then the out-projection) are port.cross_attention's output, so the recorded forward
    scores exactly what the port scores; and it records every attention block the packing names."""
    cfg, fsd, esd, batch = fixture_inputs(name)
    dcfg = configs.derive(cfg)
    ctx, _ = port.dgcnn_embed(esd, batch["extract_0"], cfg["n_neighbors"])
    N = batch["extract_1"].shape[1]
    extra = batch["extra_context"]
    ex = None if extra is None else extra.unsqueeze(1).expand(-1, N, -1)
    want = port.flow_log_prob(fsd, dcfg, batch["extract_1"][..., :dcfg["input_dim"]], ctx, ex, batch["eps"],
                              eps_cif=batch.get("eps_cif"))
    lp, rec = port_attention_maps(monkeypatch, cfg, fsd, batch["extract_1"], ctx, extra, batch["eps"], batch.get("eps_cif"),
                                  dtype=torch.float32)
    assert torch.equal(lp, want)
    assert port.cross_attention.__name__ == "cross_attention" and port.cross_attention.__module__ == "oracle.port"
    assert list(rec) == packing.attention_block_names(cfg)
    B, Nc = ctx.shape[0], ctx.shape[1]
    for w in rec.values():
        assert w.shape == (B, N, Nc)
        assert (w.sum(-1) - 1).abs().max().item() < 1e-5
