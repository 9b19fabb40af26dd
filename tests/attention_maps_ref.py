"""The oracle port's attention weights: a recorder that stands in for `oracle.port.cross_attention` and keeps, per module
prefix, the softmax weights it computes.  It restates oracle/port.py:56-63 (reference models/perceiver.py:108-115) step for
step, so the port's log-prob is unchanged while it records (tests/test_attention_maps.py checks that)."""
import torch
import torch.nn.functional as F

from flowcompare_b200 import configs
from oracle import port


def recording_cross_attention(record, keep=None):
    """A drop-in for port.cross_attention that stores w = softmax(q k^T * inner^-0.5) under record[prefix] (only prefixes in
    `keep`, when given)."""
    def cross_attention(sd, prefix, h, context):
        wq = sd[f"{prefix}.fn.attention.to_q.weight"]
        wkv = sd[f"{prefix}.fn.attention.to_kv.weight"]
        inner = wq.shape[0]
        hn = F.layer_norm(h, (h.shape[-1],), sd[f"{prefix}.norm.weight"], sd[f"{prefix}.norm.bias"], 1e-5)
        q = F.linear(hn, wq)
        kv = F.linear(context, wkv)
        k, v = kv[..., :inner], kv[..., inner:]
        w = torch.softmax(torch.matmul(q, k.transpose(1, 2)) * (inner ** -0.5), dim=-1)
        if keep is None or prefix in keep:
            record[prefix] = w.clone()
        o = torch.matmul(w, v)
        return F.linear(o, sd[f"{prefix}.fn.lin.weight"], sd[f"{prefix}.fn.lin.bias"])
    return cross_attention


def port_attention_maps(monkeypatch, cfg, flow_sd, x, context, extra=None, eps=None, eps_cif=None, dtype=torch.float64,
                        keep=None):
    """Runs port.flow_log_prob in `dtype` on CPU copies of the inputs (context: the embedding, [B,Nc,E]; extra: [B] / [B,1])
    and returns (log_prob [B,N], {prefix: weights [B,N,Nc]})."""
    record = {}
    dcfg = configs.derive(cfg)
    N = x.shape[1]
    cpu = lambda t: None if t is None else t.detach().cpu().to(dtype)
    ex = cpu(extra)
    if ex is not None:
        ex = ex.reshape(-1, 1).unsqueeze(1).expand(-1, N, -1)
    with monkeypatch.context() as m:
        m.setattr(port, "cross_attention", recording_cross_attention(record, keep))
        lp = port.flow_log_prob(port.to_dtype(flow_sd, dtype), dcfg, cpu(x)[..., :dcfg["input_dim"]], cpu(context), ex, cpu(eps),
                                eps_cif=cpu(eps_cif))
    return lp, record
