"""Packs the reference's own `state_dict`s into the device arena the C-ABI library consumes.

Input: `models_dict['flow'].state_dict()` / `models_dict['input_embedder'].state_dict()` exactly as
`load_flow` produces them (reference model_initialization.py:18-23, key layout SURVEY.md A.5) -- no
renames, no retraining.  Output per model: (header int32[], table int64[], arena fp32[]); the C++
side (`csrc/flow.cu: fc_flow_create`, `csrc/embed.cu: fc_embedder_create`) walks the table in the same
order as the code below.

Pack-time algebra (all in fp64, rounded once to fp32) -- mathematically identical to the reference:
  * every Linear weight is stored K-major `Wt[Kp][ldw]` (zero padded) so GEMM B-tiles load coalesced;
  * LayerNorm (perceiver.py:26-35) is folded into `to_q`: Wq' = Wq*diag(gamma), csum = rowsum(Wq'),
    qbias = Wq*beta, applied in the GEMM epilogue with the per-row (mu, rstd);
  * the attention out-projection `lin` (perceiver.py:95-96) and the concat `[x1 | extra | attn]`
    (transform.py:49-50, affine_coupling.py:34-35) are folded into the coupling MLP's first layer:
    W_fold = W_in[:, attn] @ W_lin, b_fold = b_in + W_in[:, attn] @ b_lin, extra/global context -> per-cloud bias;
  * ActNorm + LinearLU (act_norm.py:37-43, permuters.py:148-169) become one matrix
    W' = L U diag(exp(-log_scale)), b' = -W' shift, and their log-dets one fp64 constant;
  * the last Linear of the coupling / augment nets has its rows interleaved (s_raw_j, t_j) /
    (mean_j, log_std_j) so the elementwise epilogue sees both halves in one register tile;
  * eval-mode BatchNorm (pytorch_gcn.py:57-77) is folded into the EdgeConv [P | Q] weights.
"""
import struct

import numpy as np
import torch
import torch.nn.functional as F

from .configs import derive

FLOW_MAGIC = 0x46435F46
EMB_MAGIC = 0x46435F45
ARENA_VERSION = 2        # tensor-core weight copies as TF32 hi / lo (fp32 storage)
ARENA_VERSION_F16 = 3    # tensor-core weight copies as fp16 hi / 2^11-scaled fp16 lo
TC_FORMATS = {"tf32": ARENA_VERSION, "fp16": ARENA_VERSION_F16}


def gemm_ldw(n):
    return 64 if n <= 64 else (n + 127) // 128 * 128


def gemm_kpad(k):
    return (k + 15) // 16 * 16


# tcgen05 tiling (mirrors csrc/gemm.cuh fc_tc_*)
def tc_n_tiles(n):
    return (n + 95) // 96


def tc_bn(n):
    t = tc_n_tiles(n)
    return ((n + t - 1) // t + 15) // 16 * 16


def tc_kpad(k):
    return (k + 31) // 32 * 32


def tf32_round(x):
    """Round-to-nearest (ties away, like cvt.rna.tf32.f32) of fp32 to the 10-bit-mantissa TF32 grid."""
    i = x.contiguous().view(torch.int32)
    r = (i + 0x1000) & ~0x1FFF
    return r.view(torch.float32)


def f16_split(w32):
    """fp32 -> (hi, lo) fp16 tensors with w ~= hi + lo * 2^-11: hi = fp16(w) carries the same 11-bit significand as
    TF32, lo = fp16((w - hi) * 2^11) the next 11 bits (the scale keeps it clear of fp16's subnormal range)."""
    hi = w32.to(torch.float16)
    lo = ((w32 - hi.to(torch.float32)) * 2048.0).to(torch.float16)
    return hi, lo


class Arena:
    def __init__(self, tc_format="tf32"):
        assert tc_format in TC_FORMATS, tc_format
        self.tc_format = tc_format
        self.chunks = []
        self.size = 0
        self.table = []

    def add(self, t):
        """Appends a tensor (flattened, fp32) at a 64-float aligned offset; returns the offset."""
        t = t.detach().to(torch.float32).contiguous().reshape(-1)
        off = self.size
        pad = (-t.numel()) % 64
        self.chunks.append(t)
        if pad:
            self.chunks.append(torch.zeros(pad))
        self.size += t.numel() + pad
        return off

    def linear(self, W, b, K1, K2=0, tc=True):
        """W [N, K1+K2] (fp64 ok), b [N] or None -> table entries (w_off, b_off, whi_off, wlo_off).

        w: K-major fp32 copy for the FFMA kernel.  whi/wlo (tc=True): the same weight rounded to fp32 and
        split into TF32 hi / lo parts, [n_tiles*BN][ldk] N-major (the layout tcgen05 K-major operands and
        their TMA boxes want), for the 3xTF32 tensor-core kernel (csrc/gemm_tc.cu)."""
        N = W.shape[0]
        assert W.shape[1] == K1 + K2, (W.shape, K1, K2)
        ldw = gemm_ldw(N)
        kp1 = gemm_kpad(K1)
        kp = kp1 + (gemm_kpad(K2) if K2 else 0)
        Wt = torch.zeros(kp, ldw, dtype=torch.float64)
        Wt[:K1, :N] = W[:, :K1].t()
        if K2:
            Wt[kp1:kp1 + K2, :N] = W[:, K1:].t()
        self.table.append(self.add(Wt))
        self.table.append(self.add(b) if b is not None else -1)
        if not tc or N < 16:
            self.table.extend([-1, -1])
            return
        t1 = tc_kpad(K1)
        ldk = t1 + (tc_kpad(K2) if K2 else 0)
        rows = tc_n_tiles(N) * tc_bn(N)
        W32 = torch.zeros(rows, ldk, dtype=torch.float32)
        W32[:N, :K1] = W[:, :K1].to(torch.float32)
        if K2:
            W32[:N, t1:t1 + K2] = W[:, K1:].to(torch.float32)
        if self.tc_format == "fp16":
            hi, lo = f16_split(W32)
            assert torch.isfinite(hi.to(torch.float32)).all(), "weight beyond fp16 range: use tc_format='tf32'"
            # two fp16 per fp32 slot of the arena (bit patterns are preserved by every copy on the way to the device)
            self.table.append(self.add(hi.view(torch.float32)))
            self.table.append(self.add(lo.view(torch.float32)))
            return
        hi = tf32_round(W32)
        lo = tf32_round(W32 - hi)
        self.table.append(self.add(hi))
        self.table.append(self.add(lo))

    def vector(self, v):
        self.table.append(self.add(v))

    def finish(self):
        return torch.cat(self.chunks) if self.chunks else torch.zeros(0), np.asarray(self.table, dtype=np.int64)


def _d(sd, key):
    return sd[key].detach().to(torch.float64).cpu()


def _mlp_tensors(sd, prefix):
    hidden = []
    i = 0
    while f"{prefix}.layers.{i}.weight" in sd:
        hidden.append((_d(sd, f"{prefix}.layers.{i}.weight"), _d(sd, f"{prefix}.layers.{i}.bias")))
        i += 1
    return ((_d(sd, f"{prefix}.in_layer.weight"), _d(sd, f"{prefix}.in_layer.bias")), hidden,
            (_d(sd, f"{prefix}.out_layer.weight"), _d(sd, f"{prefix}.out_layer.bias")))


def _pack_plain_mlp(ar, sd, prefix, in_dim):
    (w_in, b_in), hidden, (w_out, b_out) = _mlp_tensors(sd, prefix)
    ar.linear(w_in, b_in, in_dim)
    for w, b in hidden:
        assert w.shape[0] == w.shape[1] == w_in.shape[0], "hidden widths must be uniform"
        ar.linear(w, b, w.shape[1])
    ar.linear(w_out, b_out, w_out.shape[1])
    return w_in.shape[0], len(hidden)


def _pack_attn(ar, sd, prefix):
    wq = _d(sd, f"{prefix}.fn.attention.to_q.weight")
    wkv = _d(sd, f"{prefix}.fn.attention.to_kv.weight")
    gamma, beta = _d(sd, f"{prefix}.norm.weight"), _d(sd, f"{prefix}.norm.bias")
    wq_f = (wq * gamma[None, :]).to(torch.float32).to(torch.float64)  # as stored
    ar.vector(wq_f.sum(dim=1))          # csum
    ar.vector(wq @ beta)                # qbias
    ar.linear(wq_f, None, wq.shape[1])
    ar.linear(wkv, None, wkv.shape[1])


def _interleave_rows(w, b):
    n = w.shape[0] // 2
    idx = torch.stack((torch.arange(n), torch.arange(n) + n), dim=1).reshape(-1)
    return w[idx], b[idx]


def _conditioner_first_layer(sd, mlp_prefix, attn_prefix, k_x, ex, is_global, E):
    """Folds [x | extra | attn/emb] first layer.  Returns (W_gemm [hid, k_x(+64)], b_fold [hid],
    w_extra [hid, ex], W_emb [hid, E] or None)."""
    w_in, b_in = _d(sd, f"{mlp_prefix}.in_layer.weight"), _d(sd, f"{mlp_prefix}.in_layer.bias")
    w_x = w_in[:, :k_x]
    w_e = w_in[:, k_x:k_x + ex]
    w_c = w_in[:, k_x + ex:]
    if attn_prefix is not None:
        w_lin, b_lin = _d(sd, f"{attn_prefix}.fn.lin.weight"), _d(sd, f"{attn_prefix}.fn.lin.bias")
        b_fold = b_in + w_c @ b_lin
        if is_global:
            # attention over N identical keys is uniform: out = lin(W_v ctx)  (SURVEY.md A.3)
            wkv = _d(sd, f"{attn_prefix}.fn.attention.to_kv.weight")
            w_v = wkv[wkv.shape[0] // 2:]
            return w_x, b_fold, w_e, w_c @ w_lin @ w_v
        return torch.cat((w_x, w_c @ w_lin), dim=1), b_fold, w_e, None
    assert is_global and w_c.shape[1] == E
    return w_x, b_in, w_e, w_c


def permuter_inverse_matrix(flow_sd, t, cfg):
    """W^-1 (fp64) of the permuter at transforms.<t>, each by the cheapest exact route: LinearLU by two triangular solves (no general
    inverse of a 300x300 product; reference models/permuters.py:171-177), Permuter by transposition (:67-69), FullCombiner by
    `inv` (:22-26), ExponentialCombiner by expm(-W) (:51-53)."""
    D = cfg["latent_dim"]
    kind = cfg["permuter_type"]
    p = f"transforms.{t}"
    eye = torch.eye(D, dtype=torch.float64)
    if kind == "LinearLU":
        lo, up = _d(flow_sd, f"{p}.lower_entries"), _d(flow_sd, f"{p}.upper_entries")
        dg = _d(flow_sd, f"{p}.unconstrained_upper_diag")
        Lm = torch.eye(D, dtype=torch.float64)
        il = np.tril_indices(D, k=-1)
        Lm[il[0], il[1]] = lo
        Um = torch.zeros(D, D, dtype=torch.float64)
        iu = np.triu_indices(D, k=1)
        Um[iu[0], iu[1]] = up
        Um[range(D), range(D)] = F.softplus(dg) + cfg["linear_lu_eps"]
        Linv = torch.linalg.solve_triangular(Lm, eye, upper=False, unitriangular=True)
        return torch.linalg.solve_triangular(Um, Linv, upper=True)
    if kind == "random_permute":
        return permuter_matrix(flow_sd, t, cfg)[0].t().contiguous()
    if kind == "FullCombiner":
        return torch.linalg.inv(_d(flow_sd, f"{p}.w"))
    if kind == "ExponentialCombiner":
        return torch.matrix_exp(-_squash(flow_sd, p, _d(flow_sd, f"{p}.w")))
    raise NotImplementedError(kind)


def fold_inverse_actnorm_lu(flow_sd, config):
    """Pack-time algebra of the inverse / sampling pass (the permuter's `.inverse` followed by reference
    models/act_norm.py:45-46, i.e. the inverse of one ActNorm + permuter pair): with the forward fold
    z' = Wp z - Wp shift, Wp = W diag(exp(-log_scale)), the inverse is z = Wp^-1 z' + shift.  Returned per pair, in
    forward layer order, as (off-diagonal part of Wp^-1, its diagonal, bias) in fp64 -- the same split the forward GEMM
    uses so that the latent's own column is applied in fp32 in the epilogue (SURVEY 8f rank 1; consumed by
    pack_flow_inverse -> csrc/flow.cu: fc_flow_sample)."""
    cfg = derive(config)
    D, L = cfg["latent_dim"], cfg["n_flow_layers"]
    out = []
    t = 1
    for layer in range(L):
        t += 1
        if layer != L - 1:
            if cfg["act_norm"]:
                shift, log_scale = _d(flow_sd, f"transforms.{t}.shift")[0], _d(flow_sd, f"transforms.{t}.log_scale")[0]
                t += 1
            else:
                shift, log_scale = torch.zeros(D, dtype=torch.float64), torch.zeros(D, dtype=torch.float64)
            Winv = torch.diag(torch.exp(log_scale)) @ permuter_inverse_matrix(flow_sd, t, cfg)
            wdiag = torch.diagonal(Winv).clone()
            out.append((Winv - torch.diag(wdiag), wdiag, shift.clone()))
            t += 1
    return out


def _coupling_prefix(cfg, layer):
    """Module prefix of flow layer `layer`'s coupling block (its CIF block for CIF flows) in the transform list of reference
    model_initialization.py:134-152: transforms.0 is the augmenter, then per layer the block, [ActNorm], permuter."""
    stride = 1 + (1 if cfg["act_norm"] else 0) + 1
    return f"transforms.{1 + layer * stride}"


def attention_block_names(config):
    """Module names of the attention blocks the flow's conditioners run over the context points, in transform order -- the
    order of the capture slots of fc_flow_attention_maps, which number the augmenter's attention 0 and layer l's l + 1 (an
    identity augmenter has none, so the list then starts at slot 1).  Empty for global-embedding flows."""
    cfg = derive(config)
    if cfg["global"]:
        return []
    cif = cfg["latent_dim"] < cfg["cif_latent_dim"]
    names = ["transforms.0.attn"] if cfg["latent_dim"] > cfg["input_dim"] else []
    for layer in range(cfg["n_flow_layers"]):
        p = _coupling_prefix(cfg, layer)
        names.append(f"{p}.flow.pre_conditioner.attn" if cif else f"{p}.pre_conditioner.attn")
    return names


INV_MAGIC = 0x46435F49


def pack_flow_inverse(flow_sd, config, tc_format="tf32"):
    """Arena of the sampling pass (csrc/flow.cu: fc_flow_set_inverse), per layer in forward order: for a CIF block the inverse of
    its (Reverse-folded) ActNorm as two per-column vectors (a = a' * isc + ibi, packing._pack_cif); for every ActNorm + permuter
    pair the off-diagonal part of Wp^-1 with bias = shift as a Linear, then its diagonal (fold_inverse_actnorm_lu)."""
    cfg = derive(config)
    ar = Arena(tc_format)
    D, L = cfg["latent_dim"], cfg["n_flow_layers"]
    cif = D < cfg["cif_latent_dim"]
    pairs = fold_inverse_actnorm_lu(flow_sd, config)
    for layer in range(L):
        if cif:
            p = _coupling_prefix(cfg, layer)
            shift, log_scale = _d(flow_sd, f"{p}.act_norm.shift")[0], _d(flow_sd, f"{p}.act_norm.log_scale")[0]
            sc = torch.exp(-log_scale).flip(0)
            bi = -shift.flip(0) * sc
            ar.vector(1.0 / sc)
            ar.vector(-bi / sc)
        if layer != L - 1:
            w_off, wdiag, shift = pairs[layer]
            ar.linear(w_off, shift, D)
            ar.vector(wdiag)
    arena, table = ar.finish()
    header = np.asarray([INV_MAGIC, TC_FORMATS[tc_format], L, D, cfg["cif_latent_dim"] if cif else 0], dtype=np.int32)
    return header, table, arena


CPL_KINDS = {"AffineCoupling": 0, "RationalQuadraticSplineCoupling": 1, "ExponentialCoupling": 2}
ACT_CODES = {"GELU": 1, "RELU": 3}   # csrc/gemm.cuh FC_ACT_*


def _squash(sd, p, w):
    """reference models/exponential_coupling.py:50 / models/permuters.py:50 (fp64)."""
    return _d(sd, f"{p}.rescale") * torch.tanh(_d(sd, f"{p}.scale") * w + _d(sd, f"{p}.shift")) + _d(sd, f"{p}.reshift") + 1e-8


def permuter_matrix(flow_sd, t, cfg):
    """(W [D,D] fp64 with z' = W z, log|det W|) of the permuter at transforms.<t> (reference model_initialization.py:117-131):
    LinearLU (permuters.py:148-169), Permuter (`random_permute`, :55-66), FullCombiner (:15-26), ExponentialCombiner (:36-52)."""
    D = cfg["latent_dim"]
    kind = cfg["permuter_type"]
    p = f"transforms.{t}"
    if kind == "LinearLU":
        lo, up = _d(flow_sd, f"{p}.lower_entries"), _d(flow_sd, f"{p}.upper_entries")
        dg = _d(flow_sd, f"{p}.unconstrained_upper_diag")
        Lm = torch.eye(D, dtype=torch.float64)
        il = np.tril_indices(D, k=-1)
        Lm[il[0], il[1]] = lo
        Um = torch.zeros(D, D, dtype=torch.float64)
        iu = np.triu_indices(D, k=1)
        Um[iu[0], iu[1]] = up
        diag = F.softplus(dg) + cfg["linear_lu_eps"]
        Um[range(D), range(D)] = diag
        return Lm @ Um, float(torch.log(diag).sum())
    if kind == "random_permute":
        perm = flow_sd[f"{p}.permutation"].long().cpu()
        W = torch.zeros(D, D, dtype=torch.float64)
        W[torch.arange(D), perm] = 1.0          # y_j = x_{perm[j]}  (index_select)
        return W, 0.0
    if kind == "FullCombiner":
        W = _d(flow_sd, f"{p}.w")
        return W, float(torch.linalg.slogdet(W)[1])
    if kind == "ExponentialCombiner":
        Wm = _squash(flow_sd, p, _d(flow_sd, f"{p}.w"))
        return torch.matrix_exp(Wm), float(torch.diagonal(Wm).sum())
    raise NotImplementedError(kind)


def _pack_cif(ar, sd, p, cfg):
    """CIF block minus its coupling (reference models/cif_block.py:50-68, :71-93).  Both `Reverse` permutations are folded away:
    with a = [x | z2] the block computes, per column j of the UN-reversed vector,
        j <  D:  a'_j = (x_j * s_{D-1-j} + t_{D-1-j} - shift_{D2-1-j}) * exp(-log_scale_{D2-1-j}),  (s, t) = affine_cif.nn(rev(z2))
        j >= D:  a'_j = (z2_j - shift_{D2-1-j}) * exp(-log_scale_{D2-1-j})
    so the affine coupling's first layer gets its input columns reversed, its last layer its s / t rows reversed (then
    interleaved for the coupling epilogue), and the ActNorm becomes a per-column (scale, bias) pair in reversed order."""
    D, D2 = cfg["latent_dim"], cfg["cif_latent_dim"]
    S = D2 - D
    for k in sd:
        if k.startswith(f"{p}.slicer.noise_dist.net."):
            assert torch.equal(sd[k], sd[k.replace(".slicer.", ".augmenter.")]), "slicer and augmenter share one net (cif_block.py:58)"
    cif_hid, n_cif = _pack_plain_mlp(ar, sd, f"{p}.augmenter.noise_dist.net", D)
    (w_in, b_in), hidden, (w_out, b_out) = _mlp_tensors(sd, f"{p}.affine_cif.nn")
    hid = w_in.shape[0]
    ar.linear(w_in.flip(1), b_in, S)
    for w, b in hidden:
        assert w.shape[0] == w.shape[1] == hid
        ar.linear(w, b, hid)
    w_o = torch.cat((w_out[:D].flip(0), w_out[D:].flip(0)), dim=0)
    b_o = torch.cat((b_out[:D].flip(0), b_out[D:].flip(0)), dim=0)
    w_o, b_o = _interleave_rows(w_o, b_o)
    ar.linear(w_o, b_o, hid)
    shift, log_scale = _d(sd, f"{p}.act_norm.shift")[0], _d(sd, f"{p}.act_norm.log_scale")[0]
    sc = torch.exp(-log_scale).flip(0)
    ar.vector(sc)
    ar.vector(-shift.flip(0) * sc)
    return cif_hid, n_cif, hid, len(hidden), float((-log_scale).sum())


def pack_flow(flow_sd, config, tc_format="tf32"):
    cfg = derive(config)
    from .spec import _check_supported
    _check_supported(cfg)
    L, D, d_in, ex = cfg["n_flow_layers"], cfg["latent_dim"], cfg["input_dim"], cfg["extra_context_dim"]
    half = D // 2
    is_global = bool(cfg["global"])
    E = cfg["input_embedding_dim"]
    inner = cfg["cross_heads"] * cfg["cross_dim_head"]
    assert inner == 64, "only inner_dim 64 (all shipped configs) is built"
    cpl_kind = CPL_KINDS[cfg["flow_type"]]
    has_aug = D > d_in
    cif = D < cfg["cif_latent_dim"]
    n2 = D - half
    cpl_out = {0: 2 * n2, 1: (cfg["num_bins_spline"] * 3 + 1) * half, 2: n2 * n2 + n2}[cpl_kind]
    ar = Arena(tc_format)
    ar.table.append(0)  # placeholder for the fp64 log-det constant
    has_cb = bool(ex) or is_global
    cb_cols, cb_bias = [], []

    def pack_conditioner(mlp_prefix, attn_prefix, k_x, out_dim, interleave=True):
        w_g, b_fold, w_e, w_emb = _conditioner_first_layer(flow_sd, mlp_prefix, attn_prefix, k_x, ex, is_global, E)
        (_, _), hidden, (w_out, b_out) = _mlp_tensors(flow_sd, mlp_prefix)
        hid = w_g.shape[0]
        ar.linear(w_g, b_fold, k_x, w_g.shape[1] - k_x)
        for w, b in hidden:
            assert w.shape[0] == w.shape[1] == hid
            ar.linear(w, b, hid)
        assert w_out.shape[0] == out_dim, (w_out.shape, out_dim)
        w_o, b_o = _interleave_rows(w_out, b_out) if interleave else (w_out, b_out)
        ar.linear(w_o, b_o, hid)
        if has_cb:
            rows = [w_e] if ex else []
            if is_global:
                rows.append(w_emb)
            cb_cols.append(torch.cat(rows, dim=1))  # [hid, Kcb]
            cb_bias.append(b_fold)
        return hid, len(hidden)

    # transforms.0 (absent -- IdentityTransform -- when latent_dim == input_dim, model_initialization.py:93-94)
    augpre_hid = n_augpre = aug_hid = n_aug = 0
    if has_aug:
        if not is_global:
            augpre_hid, n_augpre = _pack_plain_mlp(ar, flow_sd, "transforms.0.pre_attn_mlp", d_in)
            _pack_attn(ar, flow_sd, "transforms.0.attn")
        else:
            augpre_hid, n_augpre = cfg["hidden_dims"][0], len(cfg["hidden_dims"]) - 1
        aug_hid, n_aug = pack_conditioner("transforms.0.augment.noise_dist.net", "transforms.0.attn", d_in, 2 * (D - d_in))
    elif has_cb:
        # slot 0 of the per-cloud bias GEMM belongs to the augmenter: keep the slot numbering with an empty block
        hid0 = cfg["hidden_dims"][0]
        cb_cols.append(torch.zeros(hid0, ex + (E if is_global else 0), dtype=torch.float64))
        cb_bias.append(torch.zeros(hid0, dtype=torch.float64))
    cb_slot = len(ar.table)
    if has_cb:
        ar.table.extend([0, 0, -1, -1])  # (w, b, whi, wlo): w/b patched below once every layer's columns are known
    ldj_const = 0.0
    t = 1
    hid = n_hid = pre_hid = n_pre = 0
    cif_hid = n_cif = affcif_hid = n_affcif = 0
    for layer in range(L):
        p = _coupling_prefix(cfg, layer)
        if cif:
            cif_hid, n_cif, affcif_hid, n_affcif, ldj_cif = _pack_cif(ar, flow_sd, p, cfg)
            ldj_const += ldj_cif
            p = f"{p}.flow"
        if not is_global:
            pre_hid, n_pre = _pack_plain_mlp(ar, flow_sd, f"{p}.pre_conditioner.pre_attention_mlp", half)
            _pack_attn(ar, flow_sd, f"{p}.pre_conditioner.attn")
        if cpl_kind == 2:
            ar.vector(torch.cat([_d(flow_sd, f"{p}.transform.{leaf}") for leaf in ("scale", "shift", "rescale", "reshift")]))
        hid, n_hid = pack_conditioner(f"{p}.transform.nn", None if is_global else f"{p}.pre_conditioner.attn",
                                      half, cpl_out, interleave=(cpl_kind == 0))
        t += 1
        if layer != L - 1:
            if cfg["act_norm"]:
                shift, log_scale = _d(flow_sd, f"transforms.{t}.shift")[0], _d(flow_sd, f"transforms.{t}.log_scale")[0]
                t += 1
            else:
                shift, log_scale = torch.zeros(D, dtype=torch.float64), torch.zeros(D, dtype=torch.float64)
            Wperm, ldj_perm = permuter_matrix(flow_sd, t, cfg)
            Wp = Wperm @ torch.diag(torch.exp(-log_scale))
            wdiag = torch.diagonal(Wp).clone()
            ar.linear(Wp - torch.diag(wdiag), -(Wp @ shift), D)   # off-diagonal part in the GEMM ...
            ar.vector(wdiag)                                      # ... the diagonal in its epilogue (fp32, exact input)
            ldj_const += float((-log_scale).sum()) + ldj_perm
            t += 1
    if not is_global:
        pre_hid = pre_hid or cfg["pre_attention_mlp_hidden_dims"][0]
    if has_cb:
        Wcb = torch.cat(cb_cols, dim=0)  # [(L+1)*hid, Kcb]
        bcb = torch.cat(cb_bias, dim=0)
        saved = ar.table
        ar.table = []
        ar.linear(Wcb, bcb, Wcb.shape[1], tc=False)   # B rows only: always the exact fp32 kernel
        w_off, b_off = ar.table[:2]
        ar.table = saved
        ar.table[cb_slot], ar.table[cb_slot + 1] = w_off, b_off
    assert not has_aug or hid == aug_hid, "coupling and augment conditioners must share the hidden width"
    ar.table[0] = struct.unpack("<q", struct.pack("<d", ldj_const))[0]
    arena, table = ar.finish()
    clamp = cfg["clamp_dist"] if cif and cfg["clamp_dist"] else 0.0
    clamp_bits = struct.unpack("<i", struct.pack("<f", float(clamp)))[0]
    header = np.asarray([FLOW_MAGIC, TC_FORMATS[tc_format], L, D, d_in, half, ex, int(is_global), E, inner,
                         cfg["attn_input_dim"], hid, n_hid, pre_hid or 0, n_pre, aug_hid, n_aug,
                         augpre_hid, n_augpre,
                         cpl_kind, cfg["num_bins_spline"], ACT_CODES[cfg["coupling_block_nonlinearity"]], int(has_aug),
                         cfg["cif_latent_dim"] if cif else 0, cif_hid, n_cif, affcif_hid, n_affcif, clamp_bits], dtype=np.int32)
    return header, table, arena


def _bn_fold(sd, prefix):
    w, b = _d(sd, f"{prefix}.weight"), _d(sd, f"{prefix}.bias")
    rm, rv = _d(sd, f"{prefix}.running_mean"), _d(sd, f"{prefix}.running_var")
    a = w / torch.sqrt(rv + 1e-5)
    return a, b - a * rm


def pack_embedder(emb_sd, config, tc_format="tf32"):
    cfg = derive(config)
    name = cfg["input_embedder"]
    if name == "PAConv":
        from .paconv_packing import pack_paconv
        return pack_paconv(emb_sd, cfg, tc_format)
    if name not in ("DGCNNembedder", "DGCNNembedderGlobal"):
        raise NotImplementedError(name)
    kind = 1 if name == "DGCNNembedderGlobal" else 0
    ar = Arena(tc_format)
    cins = [cfg["input_dim"], 64, 64, 128]
    for i in range(4):
        W = _d(emb_sd, f"conv{i + 1}.0.weight")[:, :, 0, 0]
        cin = cins[i]
        assert W.shape[1] == 2 * cin, (W.shape, cin)
        a, b = _bn_fold(emb_sd, f"bn{i + 1}")
        w1, w2 = W[:, :cin], W[:, cin:]
        Wpq = torch.cat((a[:, None] * w1, a[:, None] * (w2 - w1)), dim=0)
        bpq = torch.cat((torch.zeros_like(b), b), dim=0)
        ar.linear(Wpq, bpq, cin, tc=False)   # feeds the bit-exact kNN of the next block: exact fp32 only
    W5 = _d(emb_sd, "conv5.0.weight")[:, :, 0]
    a5, b5 = _bn_fold(emb_sd, "bn5")
    ar.linear(a5[:, None] * W5, b5, 512)
    out_hid, n_out = _pack_plain_mlp(ar, emb_sd, "out_mlp", 1024 if kind == 1 else 512)
    arena, table = ar.finish()
    header = np.asarray([EMB_MAGIC, TC_FORMATS[tc_format], kind, cfg["input_dim"], cfg["n_neighbors"],
                         cfg["input_embedding_dim"], out_hid, n_out], dtype=np.int32)
    return header, table, arena


GRAD_MAGIC = 0x46435F47


def grad_unsupported_transform(config):
    """The transform of this flow the input-gradient pass has no backward for (reference class name), or None."""
    cfg = derive(config)
    if cfg["latent_dim"] < cfg["cif_latent_dim"]:
        return "CIFblock"
    if cfg["flow_type"] != "AffineCoupling":
        return cfg["flow_type"]
    return None


def _pack_mlp_t(ar, w_first, k_x, hidden, w_out, has_o):
    """An MLP's backward contractions as Linears with the transposed weights: the first layer's x columns, its attention-output
    columns (`has_o`), the hidden layers, the out layer (rows as the forward stores them)."""
    ar.linear(w_first[:, :k_x].t(), None, w_first.shape[0])
    if has_o:
        ar.linear(w_first[:, k_x:].t(), None, w_first.shape[0])
    for w, _ in hidden:
        ar.linear(w.t(), None, w.shape[0])
    ar.linear(w_out.t(), None, w_out.shape[0])


def pack_flow_grad(flow_sd, config):
    """Arena of the input-gradient pass (csrc/flow.cu: fc_flow_set_grad): the transpose W^T of every folded matrix the forward pass
    runs, in the forward's order -- per conditioner the pre-attention MLP, to_q with the LayerNorm gain folded in (Wq diag(gamma)),
    the coupling (augment) MLP with its first layer split into the x columns and the attention-output columns (out-projection
    folded in), and the off-diagonal part of ActNorm + permuter.  Every backward contraction dX = dY W is then an ordinary Linear
    with weight W^T.  The tensor-core copies are always 3xTF32 (fp32 exponent range): gradients are not bounded a priori, and the
    3xFP16 format would turn values beyond fp16's range into NaN rows."""
    cfg = derive(config)
    bad = grad_unsupported_transform(cfg)
    if bad is not None:
        raise NotImplementedError(f"input gradients: no backward pass for {bad}")
    L, D, d_in, ex = cfg["n_flow_layers"], cfg["latent_dim"], cfg["input_dim"], cfg["extra_context_dim"]
    half = D // 2
    is_global = bool(cfg["global"])
    E = cfg["input_embedding_dim"]
    ar = Arena("tf32")

    def conditioner(pre_prefix, attn_prefix, mlp_prefix, k_x, fold_prefix):
        if not is_global:
            (w_in, _), hidden, (w_out, _) = _mlp_tensors(flow_sd, pre_prefix)
            _pack_mlp_t(ar, w_in, k_x, hidden, w_out, False)
            wq = _d(flow_sd, f"{attn_prefix}.fn.attention.to_q.weight")
            gamma = _d(flow_sd, f"{attn_prefix}.norm.weight")
            wq_f = (wq * gamma[None, :]).to(torch.float32).to(torch.float64)     # as pack_flow stores it
            ar.linear(wq_f.t(), None, wq_f.shape[0])
        w_g, _, _, _ = _conditioner_first_layer(flow_sd, mlp_prefix, fold_prefix, k_x, ex, is_global, E)   # as pack_flow folds it
        (_, _), hidden, (w_out, b_out) = _mlp_tensors(flow_sd, mlp_prefix)
        w_o, _ = _interleave_rows(w_out, b_out)
        _pack_mlp_t(ar, w_g, k_x, hidden, w_o, not is_global)

    if D > d_in:
        conditioner("transforms.0.pre_attn_mlp", "transforms.0.attn", "transforms.0.augment.noise_dist.net", d_in,
                    "transforms.0.attn")
    t = 1
    for layer in range(L):
        p = _coupling_prefix(cfg, layer)
        conditioner(f"{p}.pre_conditioner.pre_attention_mlp", f"{p}.pre_conditioner.attn", f"{p}.transform.nn", half,
                    None if is_global else f"{p}.pre_conditioner.attn")
        t += 1
        if layer != L - 1:
            if cfg["act_norm"]:
                log_scale = _d(flow_sd, f"transforms.{t}.log_scale")[0]
                t += 1
            else:
                log_scale = torch.zeros(D, dtype=torch.float64)
            Wp = permuter_matrix(flow_sd, t, cfg)[0] @ torch.diag(torch.exp(-log_scale))
            ar.linear((Wp - torch.diag(torch.diagonal(Wp))).t(), None, D)
            t += 1
    arena, table = ar.finish()
    header = np.asarray([GRAD_MAGIC, ARENA_VERSION, L, D], dtype=np.int32)
    return header, table, arena
