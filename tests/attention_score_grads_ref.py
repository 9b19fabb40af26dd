"""fp64 reference of the attention score gradients (engine.attention_score_grads): a recorder that stands in for
`oracle.port.cross_attention`, restating oracle/port.py:56-63 (reference models/perceiver.py:108-115) step for step, keeps each
block's scores `sim` with `retain_grad()`, and `lp.sum().backward()` through `port.flow_log_prob` with eps fixed -- the
reference's `sim.grad`.  A point's log-prob depends on its own query row only, so sim.grad[b, i, j] = d lp[b, i] / d s_ij."""
import torch
import torch.nn.functional as F

from flowcompare_b200 import configs
from oracle import port


def recording_cross_attention(record, bias=None):
    """A drop-in for port.cross_attention that stores, under record[prefix], the scores `sim` (gradient retained), the weights
    `P`, the values `v` and the attention output `o` (gradient retained).  bias = (prefix, j, h): h added to column j of that
    block's scores, for every cloud and query row (the rows are scored independently)."""
    def cross_attention(sd, prefix, h, context):
        wq = sd[f"{prefix}.fn.attention.to_q.weight"]
        wkv = sd[f"{prefix}.fn.attention.to_kv.weight"]
        inner = wq.shape[0]
        hn = F.layer_norm(h, (h.shape[-1],), sd[f"{prefix}.norm.weight"], sd[f"{prefix}.norm.bias"], 1e-5)
        q = F.linear(hn, wq)
        kv = F.linear(context, wkv)
        k, v = kv[..., :inner], kv[..., inner:]
        sim = torch.matmul(q, k.transpose(1, 2)) * (inner ** -0.5)
        if bias is not None and bias[0] == prefix:
            shift = torch.zeros_like(sim)
            shift[..., bias[1]] = bias[2]
            sim = sim + shift
        w = torch.softmax(sim, dim=-1)
        o = torch.matmul(w, v)
        if sim.requires_grad:
            sim.retain_grad()
            o.retain_grad()
        record[prefix] = {"sim": sim, "P": w, "v": v, "o": o}
        return F.linear(o, sd[f"{prefix}.fn.lin.weight"], sd[f"{prefix}.fn.lin.bias"])
    return cross_attention


def port_score_grads(monkeypatch, cfg, flow_sd, x, context, extra=None, eps=None, dtype=torch.float64, bias=None, backward=True):
    """Runs port.flow_log_prob in `dtype` on CPU copies of the inputs (context: the embedding [B,Nc,E]; extra [B] / [B,1]) with x
    requiring grad, then (backward) lp.sum().backward().  Returns (log_prob [B,N], {prefix: {"sim", "P", "v", "o"}}): after the
    backward, record[prefix]["sim"].grad is that block's d lp_i / d s_ij [B,N,Nc] and record[prefix]["o"].grad its dL/do."""
    record = {}
    dcfg = configs.derive(cfg)
    cpu = lambda t: None if t is None else t.detach().cpu().to(dtype)
    N = x.shape[1]
    ex = cpu(extra)
    if ex is not None:
        ex = ex.reshape(-1, 1).unsqueeze(1).expand(-1, N, -1)
    with monkeypatch.context() as m, torch.enable_grad():
        m.setattr(port, "cross_attention", recording_cross_attention(record, bias))
        xv = cpu(x)[..., :dcfg["input_dim"]].clone().requires_grad_(True)
        lp = port.flow_log_prob(port.to_dtype(flow_sd, dtype), dcfg, xv, cpu(context), ex, cpu(eps))
        if backward:
            lp.sum().backward()
    return lp.detach(), record


def score_grads(record):
    """{prefix: d lp_i / d s_ij [B,N,Nc]} of a recorded backward."""
    return {p: r["sim"].grad for p, r in record.items()}


def closed_form(r):
    """P (dO.v - dO.o) from a recorded block: the formula the CUDA kernel evaluates."""
    dO = r["o"].grad
    dp = torch.matmul(dO, r["v"].transpose(1, 2))
    D = (dO * r["o"]).sum(-1, keepdim=True)
    return r["P"].detach() * (dp - D.detach())


def row_error(got, want, floor_frac=1e-6):
    """Per query row: max_j |got - want| / max_j |want|, the normaliser floored at floor_frac * max |want| of the block (rows
    whose gradient is within fp32 noise of zero would otherwise divide by ~0).  [B*n_query] float64."""
    got = got.detach().cpu().double().reshape(-1, want.shape[-1])
    want = want.detach().double().reshape(-1, want.shape[-1])
    scale = want.abs().amax(-1).clamp_min(floor_frac * want.abs().max().item())
    return (got - want).abs().amax(-1) / scale
