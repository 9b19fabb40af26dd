"""fp64 reference of the importance-weighted log-likelihood (engine.log_prob_iw): `oracle.port.flow_log_prob` once per
augmentation draw in float64, then the fp64 logmeanexp over the draws, with the NaN / inf rules `fc_logmeanexp` follows."""
import math

import numpy as np
import torch

from flowcompare_b200 import configs
from oracle import port


def logmeanexp(draws):
    """log((1/K) sum_k exp(draws[k])) over the leading axis in float64.  NaN if any draw is NaN, +inf if any is +inf (and none
    is NaN); -inf draws drop out of the sum, all -inf gives -inf."""
    d = np.asarray(torch.as_tensor(draws).double().cpu().numpy(), dtype=np.float64)
    K = d.shape[0]
    nan = np.isnan(d).any(axis=0)
    pinf = (d == np.inf).any(axis=0)
    m = np.max(np.where(np.isnan(d), -np.inf, d), axis=0)
    finite = np.isfinite(m)
    ms = np.where(finite, m, 0.0)
    s = np.exp(np.where(np.isnan(d), -np.inf, d) - ms).sum(axis=0)
    with np.errstate(divide="ignore"):
        out = np.where(finite, ms + np.log(s) - math.log(K), m)
    out = np.where(pinf, np.inf, out)
    out = np.where(nan, np.nan, out)
    return torch.from_numpy(out)


def port_log_prob_iw(cfg, fsd, x, ctx, extra, eps, eps_cif=None, dtype=torch.float64):
    """(IW [B,N], draws [K,B,N]) from the port in `dtype` on CPU copies: ctx is the embedding [B,Nc,E] (or [B,E] for the global
    embedder), extra [B] / [B,1] or None, eps [K,B,N,latent-input_dim], eps_cif [K,L,B,N,S] or None."""
    dcfg = configs.derive(cfg)
    cpu = lambda t: None if t is None else t.detach().cpu().to(dtype)
    x = cpu(x)[..., :dcfg["input_dim"]]
    N = x.shape[1]
    c = cpu(ctx)
    if c.dim() == 2:      # global embedding: the port takes it repeated per point, as the reference does
        c = c.unsqueeze(1).expand(-1, N, -1)
    ex = cpu(extra)
    if ex is not None:
        ex = ex.reshape(-1, 1).unsqueeze(1).expand(-1, N, -1)
    sd = port.to_dtype(fsd, dtype)
    eps, eps_cif = cpu(eps), cpu(eps_cif)
    draws = torch.stack([port.flow_log_prob(sd, dcfg, x, c, ex, eps[k], eps_cif=None if eps_cif is None else eps_cif[k])
                         for k in range(eps.shape[0])])
    return logmeanexp(draws), draws
