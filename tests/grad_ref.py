"""fp64 reference of the input gradients (engine.log_prob_grad): autograd of `oracle.port.flow_log_prob` with respect to x, eps
held fixed -- what `torch.autograd.grad(flow.log_prob(x, context=...).sum(), x)` gives on the reference.  Also the table walkers
that read a packed Linear back out of the forward arena (packing.pack_flow) and the input-gradient arena (packing.pack_flow_grad),
in the order csrc/flow.cu (fc_flow_create, fc_flow_set_grad) reads them."""
import torch

from flowcompare_b200 import configs, packing
from oracle import port


def port_log_prob_grad(cfg, fsd, x, ctx, extra, eps, dtype=torch.float64):
    """(log_prob [B,N], grad [B,N,input_dim]) from the port in `dtype` on CPU copies: ctx is the embedding [B,Nc,E] (or [B,E] for the
    global embedder), extra [B] / [B,1] or None, eps [B,N,latent-input_dim]."""
    dcfg = configs.derive(cfg)
    cpu = lambda t: None if t is None else t.detach().cpu().to(dtype)
    with torch.enable_grad():
        xv = cpu(x)[..., :dcfg["input_dim"]].clone().requires_grad_(True)
        N = xv.shape[1]
        c = cpu(ctx)
        if c.dim() == 2:      # global embedding: the port takes it repeated per point, as the reference does
            c = c.unsqueeze(1).expand(-1, N, -1)
        ex = cpu(extra)
        if ex is not None:
            ex = ex.reshape(-1, 1).unsqueeze(1).expand(-1, N, -1)
        lp = port.flow_log_prob(port.to_dtype(fsd, dtype), dcfg, xv, c, ex, cpu(eps))
        (g,) = torch.autograd.grad(lp.sum(), xv)
    return lp.detach(), g


def grad_error(got, want):
    """Per point: max_c |got - want| / max(1, max_c |want|) -- [B*N] float64."""
    got, want = got.detach().cpu().double().reshape(-1, want.shape[-1]), want.double().reshape(-1, want.shape[-1])
    return (got - want).abs().amax(-1) / want.abs().amax(-1).clamp_min(1.0)


def dense_linear(arena, w_off, K1, K2, N):
    """W [N, K1+K2] of a Linear packed K-major at float offset w_off (packing.Arena.linear)."""
    ldw = packing.gemm_ldw(N)
    kp1 = packing.gemm_kpad(K1)
    kp = kp1 + (packing.gemm_kpad(K2) if K2 else 0)
    Wt = arena[w_off:w_off + kp * ldw].reshape(kp, ldw)
    cols = [Wt[:K1, :N]] + ([Wt[kp1:kp1 + K2, :N]] if K2 else [])
    return torch.cat(cols, dim=0).t()


class _Walk:
    def __init__(self, table, pos):
        self.table, self.pos, self.out = table, pos, {}

    def linear(self, name, K1, K2, N):
        self.out[name] = (int(self.table[self.pos]), K1, K2, N)
        self.pos += 4

    def skip(self, n=1):
        self.pos += n

    def mlp(self, name, K1, K2, hid, n_hidden, N_out):
        self.linear(f"{name}.in", K1, K2, hid)
        for i in range(n_hidden):
            self.linear(f"{name}.hidden{i}", hid, 0, hid)
        self.linear(f"{name}.out", hid, 0, N_out)


def forward_linears(header, table):
    """{name: (w_off, K1, K2, N)} of the forward arena of an affine-coupling flow without CIF blocks."""
    (L, D, d_in, half, ex, is_global, E, inner, attn_in, hid, n_hid, pre_hid, n_pre, aug_hid, n_aug, augpre_hid,
     n_augpre) = [int(v) for v in header[2:19]]
    has_aug = int(header[22])
    w = _Walk(table, 1)
    k2 = 0 if is_global else inner
    if has_aug:
        if not is_global:
            w.mlp("aug.pre", d_in, 0, augpre_hid, n_augpre, attn_in)
            w.skip(2)
            w.linear("aug.q", attn_in, 0, inner)
            w.linear("aug.kv", E, 0, 2 * inner)
        w.mlp("aug.cpl", d_in, k2, aug_hid, n_aug, 2 * (D - d_in))
    if ex or is_global:
        w.skip(4)
    for l in range(L):
        if not is_global:
            w.mlp(f"{l}.pre", half, 0, pre_hid, n_pre, attn_in)
            w.skip(2)
            w.linear(f"{l}.q", attn_in, 0, inner)
            w.linear(f"{l}.kv", E, 0, 2 * inner)
        w.mlp(f"{l}.cpl", half, k2, hid, n_hid, 2 * (D - half))
        if l != L - 1:
            w.linear(f"{l}.lu", D, 0, D)
            w.skip(1)
    assert w.pos == len(table)
    return w.out


def grad_linears(fwd_header, table):
    """{name: (w_off, K1, K2, N)} of the input-gradient arena (the order of fc_flow_set_grad)."""
    (L, D, d_in, half, ex, is_global, E, inner, attn_in, hid, n_hid, pre_hid, n_pre, aug_hid, n_aug, augpre_hid,
     n_augpre) = [int(v) for v in fwd_header[2:19]]
    has_aug = int(fwd_header[22])
    w = _Walk(table, 0)

    def mlp_t(name, k_x, has_o, hid_, n_hidden, n_out):
        w.linear(f"{name}.in_x", hid_, 0, k_x)
        if has_o:
            w.linear(f"{name}.in_o", hid_, 0, inner)
        for i in range(n_hidden):
            w.linear(f"{name}.hidden{i}", hid_, 0, hid_)
        w.linear(f"{name}.out", n_out, 0, hid_)

    if has_aug:
        if not is_global:
            mlp_t("aug.pre", d_in, False, augpre_hid, n_augpre, attn_in)
            w.linear("aug.q", inner, 0, attn_in)
        mlp_t("aug.cpl", d_in, not is_global, aug_hid, n_aug, 2 * (D - d_in))
    for l in range(L):
        if not is_global:
            mlp_t(f"{l}.pre", half, False, pre_hid, n_pre, attn_in)
            w.linear(f"{l}.q", inner, 0, attn_in)
        mlp_t(f"{l}.cpl", half, not is_global, hid, n_hid, 2 * (D - half))
        if l != L - 1:
            w.linear(f"{l}.lu", D, 0, D)
    assert w.pos == len(table)
    return w.out
