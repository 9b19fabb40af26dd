"""Host side of the drop-in: mirrors the reference's `model_dict` / `inner_loop` interface.

    models_dict = initialize_flow(config, device, 'test')      # reference, unchanged
    models_dict = load_flow(checkpoint, models_dict)            # reference, unchanged
    engine = FlowCompareB200(models_dict, config)               # packs the state_dicts once
    loss, log_prob, bpd = engine.inner_loop(batch)              # == inner_loop(batch, models_dict, config)

or `accelerate(models_dict, config)` which returns a models_dict whose 'flow' / 'input_embedder'
entries are adapters with the reference call signatures (`flow.log_prob(x, context=, extra_context=)`,
`input_embedder(extract_0)`), so the reference's own `inner_loop` / `test_flow.evaluate_on_test` run
unmodified on top of the CUDA path.

PyTorch is used for device memory and streams only; every computation is a call into
`libflowcompare_b200.so`.  There is no CPU path: tensors must live on a CUDA device (host tensors are
copied there), and a missing library raises.
"""
import math

import numpy as np
import torch

from . import lib as _lib
from . import packing
from .configs import derive


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f32c(t, device):
    return t.to(device=device, dtype=torch.float32).contiguous()


IW_MAX_PASS_ROWS = 1 << 20      # rows (draws x points) of one fc_flow_log_prob_draws pass
GRAD_MAX_PASS_ROWS = 1 << 16    # points of one fc_flow_log_prob_grad pass (11.8 GB of workspace at the shipped widths)


def _check_shape(what, name, t, shape):
    if tuple(t.shape) != tuple(shape):
        raise _lib.FlowCompareError(f"{what}: {name} must be {list(shape)}, got {list(t.shape)}")


def _n_draws(n, what):
    if isinstance(n, bool) or not isinstance(n, (int, np.integer)) or n < 1:
        raise _lib.FlowCompareError(f"{what}: the number of draws must be a positive int, got {n!r}")
    return int(n)


class FlowCompareB200:
    """Per-point conditional log-likelihood engine (eval mode only).

    Parameters: `models` -- the reference's `models_dict` ({'flow': Flow, 'input_embedder': Module}) or a
    pair of state_dicts `(flow_sd, embedder_sd)`; `config` -- the reference config dict (YAML values).
    `precision`: 'fp32' (exact FFMA GEMMs), 'tf32x3' (tcgen05 tensor cores, 3xTF32 error-compensated) or 'fp16x3'
    (tcgen05, 3xFP16 error-compensated: the same 11-bit significands at twice the tensor rate; activations beyond
    fp16's range, |a| >= 65520, turn the affected rows into NaN instead of a silently wrong value).
    """

    def __init__(self, models, config, device="cuda:0", precision="fp32"):
        self.lib = _lib.load()
        self.config = derive(config)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.FlowCompareError("flowcompare_b200 runs on CUDA devices only (no CPU fallback)")
        self.precision_name = precision
        self.precision, tc_format = _lib.PRECISIONS[precision]
        if isinstance(models, dict):
            for m in (models["flow"], models["input_embedder"]):
                if getattr(m, "training", False):
                    raise _lib.FlowCompareError("train-mode modules (BN / ActNorm data init) are out of scope: call .eval()")
            flow_sd, emb_sd = models["flow"].state_dict(), models["input_embedder"].state_dict()
        else:
            flow_sd, emb_sd = models
        self.d_in = self.config["input_dim"]
        self.D = self.config["latent_dim"]
        self.E = self.config["input_embedding_dim"]
        self.is_global = bool(self.config["global"])
        self.has_extra = bool(self.config["using_extra_context"])
        self.k = self.config["n_neighbors"]
        self.L = self.config["n_flow_layers"]
        # CIF blocks (latent_dim < cif_latent_dim, reference models/cif_block.py:30-37) draw their own noise
        self.cif_S = max(0, self.config["cif_latent_dim"] - self.D)
        with torch.cuda.device(self.device):
            self._flow = self._create(packing.pack_flow(flow_sd, self.config, tc_format), self.lib.fc_flow_create,
                                      "fc_flow_create")
            self._emb = self._create(packing.pack_embedder(emb_sd, self.config, tc_format), self.lib.fc_embedder_create,
                                     "fc_embedder_create")
        self._ws = None
        self._seed_counter = 0
        self._tc_format = tc_format
        self._flow_sd_for_inverse = flow_sd      # the inverse ActNorm+LinearLU matrices are packed on the first make_sample
        self._inv = None
        self._grad = None                        # the transposed weights of log_prob_grad are packed on its first call
        # reference Flow(sample_dist=Normal(loc, scale)) (model_initialization.py:154-161): buffers of the flow's state_dict
        self._sample_loc = float(flow_sd["sample_dist.loc"].reshape(-1)[0]) if "sample_dist.loc" in flow_sd else 0.0
        self._sample_scale = float(flow_sd["sample_dist.scale"].reshape(-1)[0]) if "sample_dist.scale" in flow_sd else 1.0

    # ------------------------------------------------------------------ lifecycle
    def _create(self, packed, create_fn, what):
        header, table, arena = packed
        arena_dev = arena.to(self.device)
        handle = _lib.c_vp()
        rc = create_fn(header.ctypes.data, len(header), table.ctypes.data, len(table), arena_dev.data_ptr(),
                       arena_dev.numel(), handle)
        _lib.check(rc, what)
        return {"handle": handle, "arena": arena_dev, "header": header, "table": table}

    def close(self):
        if getattr(self, "_flow", None):
            self.lib.fc_flow_destroy(self._flow["handle"])
            self._flow = None
        if getattr(self, "_emb", None):
            self.lib.fc_embedder_destroy(self._emb["handle"])
            self._emb = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def weight_bytes(self):
        return 4 * (self._flow["arena"].numel() + self._emb["arena"].numel())

    def _workspace(self, nbytes):
        if nbytes < 0:
            _lib.check(int(nbytes), "workspace query")
        if self._ws is None or self._ws.numel() < nbytes + 256:     # + 256: room to round the base up to the ABI's alignment
            self._ws = None
            self._ws = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=self.device)
        base = self._ws.data_ptr()
        return (base + 255) // 256 * 256

    # ------------------------------------------------------------------ pieces
    def embed(self, extract_0, return_knn=False):
        """`input_embedder(extract_0)`: [B,Nc,>=input_dim] -> [B,Nc,E] (or [B,E] for the global embedder)."""
        with torch.cuda.device(self.device):
            pts = _f32c(extract_0[:, :, :self.d_in], self.device)
            B, Nc = pts.shape[0], pts.shape[1]
            out = torch.empty((B, self.E) if self.is_global else (B, Nc, self.E), dtype=torch.float32, device=self.device)
            idx = None
            if return_knn:
                idx = torch.empty((4, B, Nc, self.k), dtype=torch.int32, device=self.device)
            nbytes = self.lib.fc_embedder_workspace_bytes(self._emb["handle"], B, Nc)
            ws = self._workspace(nbytes)
            rc = self.lib.fc_embed(self._emb["handle"], pts.data_ptr(), out.data_ptr(), B, Nc, _ptr(idx), ws, nbytes,
                                   self.precision, _stream())
            _lib.check(rc, "fc_embed")
        return (out, idx) if return_knn else out

    def _next_seed(self):
        """Default noise seeds follow torch's global seed (like the reference's `Normal.rsample`, `torch.manual_seed` makes
        a run reproducible) and differ per device and per call, so ranks / engines do not score their pairs with the same
        noise."""
        self._seed_counter += 1
        dev = self.device.index if self.device.index is not None else torch.cuda.current_device()
        return (torch.initial_seed() * 0x9E3779B1 + dev * 0x85EBCA6B + self._seed_counter) & 0x7FFFFFFFFFFFFFFF

    def draw_eps(self, B, N, seed=None):
        """Device-side N(0,1) draw for the augmentation noise (reference: models/distributions.py:148-153)."""
        with torch.cuda.device(self.device):
            eps = torch.empty((B, N, self.D - self.d_in), dtype=torch.float32, device=self.device)
            if seed is None:
                seed = self._next_seed()
            _lib.check(self.lib.fc_fill_normal(eps.data_ptr(), eps.numel(), seed, 0, _stream()), "fc_fill_normal")
        return eps

    def draw_eps_cif(self, B, N, seed=None):
        """The CIF blocks' draws [L, B, N, cif_latent_dim - latent_dim] (reference models/cif_block.py:74), on the device."""
        with torch.cuda.device(self.device):
            eps = torch.empty((self.L, B, N, self.cif_S), dtype=torch.float32, device=self.device)
            if seed is None:
                seed = self._next_seed()
            _lib.check(self.lib.fc_fill_normal(eps.data_ptr(), eps.numel(), seed, 1 << 40, _stream()), "fc_fill_normal")
        return eps

    def log_prob(self, x, context, extra_context=None, eps=None, eps_cif=None):
        """`Flow.log_prob(x, context=, extra_context=)` (reference models/transform.py:70-76).

        x [B,N,input_dim]; context [B,Nc,E] (or [B,E] / repeated [B,N,E] for the global embedder);
        extra_context [B], [B,1] or the repeated [B,N,1] the reference passes; eps [B,N,latent-input_dim]
        optional (default: drawn on the device); eps_cif [L,B,N,cif_latent_dim-latent_dim] likewise, CIF flows only."""
        with torch.cuda.device(self.device):
            x, context, Nc, extra, eps, eps_cif = self._flow_inputs("log_prob", x, context, extra_context, eps, eps_cif)
            B, N = x.shape[0], x.shape[1]
            out = torch.empty((B, N), dtype=torch.float32, device=self.device)
            nbytes = self.lib.fc_flow_workspace_bytes(self._flow["handle"], B, N, Nc)
            ws = self._workspace(nbytes)
            if self.cif_S:
                rc = self.lib.fc_flow_log_prob_cif(self._flow["handle"], x.data_ptr(), context.data_ptr(), _ptr(extra),
                                                   _ptr(eps), eps_cif.data_ptr(), out.data_ptr(), B, N, Nc, ws, nbytes,
                                                   self.precision, _stream())
                _lib.check(rc, "fc_flow_log_prob_cif")
            else:
                rc = self.lib.fc_flow_log_prob(self._flow["handle"], x.data_ptr(), context.data_ptr(), _ptr(extra),
                                               _ptr(eps), out.data_ptr(), B, N, Nc, ws, nbytes, self.precision, _stream())
                _lib.check(rc, "fc_flow_log_prob")
        return out

    def log_prob_iw(self, x, context, extra_context=None, n_draws=8, eps=None, eps_cif=None, return_draws=False,
                    draws_per_pass=None, workspace_budget=None):
        """Importance-weighted log p(x | context) over `n_draws` augmentation draws:
        IW_K = log((1/K) sum_k exp(lp_k)), lp_k = `log_prob(x, context, eps=eps[k])`.

        `log_prob` is a single-sample estimate: the augmenter's noise dims (and every CIF block's) are drawn from q(e | x, c), so
        exp(lp_k) is an unbiased estimate of p(x | c) and lp_k itself is noisy.  IW_K is never below the mean of its draws and
        approaches log p(x | c) as K grows; K = 1 is exactly the reference's `Flow.log_prob`.
        Arguments as `log_prob` (`context` is the embedding); eps [K,B,N,latent-input_dim] and eps_cif
        [K,L,B,N,cif_latent_dim-latent_dim] (CIF flows) optional, drawn on the device by default.  The draws run in passes of at
        most 2^20 rows (K_pass*B*N), fewer with `draws_per_pass` or when a pass's workspace would exceed `workspace_budget`
        bytes; the result does not depend on the split.  Returns IW [B,N], or (IW, draws [K,B,N]) with `return_draws`:
        draws[k] is bitwise `log_prob(x, context, eps=eps[k], eps_cif=eps_cif[k])`."""
        K = _n_draws(n_draws, "log_prob_iw")
        if draws_per_pass is not None:
            _n_draws(draws_per_pass, "log_prob_iw: draws_per_pass")
        with torch.cuda.device(self.device):
            x = _f32c(x[..., :self.d_in], self.device)
            B, N = x.shape[0], x.shape[1]
            context, Nc, extra = self._prep_context(context, extra_context, B)
            S = self.D - self.d_in
            if eps is not None:
                eps = _f32c(eps, self.device)
                _check_shape("log_prob_iw", "eps", eps, (K, B, N, S))
            if eps_cif is not None:
                if not self.cif_S:
                    raise _lib.FlowCompareError("log_prob_iw: eps_cif given but this flow has no CIF blocks")
                eps_cif = _f32c(eps_cif, self.device)
                _check_shape("log_prob_iw", "eps_cif", eps_cif, (K, self.L, B, N, self.cif_S))
            deterministic = S == 0 and not self.cif_S       # every draw is the same log_prob: one pass
            if N > IW_MAX_PASS_ROWS:
                raise _lib.FlowCompareError(f"log_prob_iw: {N} points per cloud exceed one pass of {IW_MAX_PASS_ROWS} rows")
            h = self._flow["handle"]
            wsb = lambda bc, kp: self.lib.fc_flow_log_prob_draws_workspace_bytes(h, bc, N, Nc, kp)
            bc = min(B, IW_MAX_PASS_ROWS // N)                                  # clouds per pass
            kp = K if deterministic else max(1, min(K, IW_MAX_PASS_ROWS // (bc * N)))   # draws per pass
            if draws_per_pass is not None and not deterministic:
                kp = min(kp, int(draws_per_pass))
            if workspace_budget is not None:
                while not deterministic and kp > 1 and wsb(bc, kp) > workspace_budget:
                    kp -= 1
                while bc > 1 and wsb(bc, kp) > workspace_budget:
                    bc = (bc + 1) // 2
            draws = torch.empty((K, B, N), dtype=torch.float32, device=self.device)
            for b0 in range(0, B, bc):
                b1 = min(B, b0 + bc)
                nb = b1 - b0
                for k0 in range(0, K, kp):
                    k1 = min(K, k0 + kp)
                    nk = k1 - k0
                    pe = pc = None
                    if S and not deterministic:
                        if eps is None:
                            pe = torch.empty((nk, nb, N, S), dtype=torch.float32, device=self.device)
                            _lib.check(self.lib.fc_fill_normal(pe.data_ptr(), pe.numel(), self._next_seed(), 0, _stream()),
                                       "fc_fill_normal")
                        else:
                            pe = eps[k0:k1, b0:b1].contiguous()
                    if self.cif_S:
                        if eps_cif is None:   # iid draws: the layout [L, B, K, N, S] the pass reads needs no permute
                            pc = torch.empty((self.L, nb, nk, N, self.cif_S), dtype=torch.float32, device=self.device)
                            _lib.check(self.lib.fc_fill_normal(pc.data_ptr(), pc.numel(), self._next_seed(), 1 << 40, _stream()),
                                       "fc_fill_normal")
                        else:
                            pc = eps_cif[k0:k1, :, b0:b1].permute(1, 2, 0, 3, 4).contiguous()
                    out = draws[k0:k1] if nb == B else torch.empty((nk, nb, N), dtype=torch.float32, device=self.device)
                    nbytes = wsb(nb, nk)
                    ws = self._workspace(nbytes)
                    rc = self.lib.fc_flow_log_prob_draws(h, x[b0:b1].data_ptr(), context[b0:b1].data_ptr(),
                                                         _ptr(None if extra is None else extra[b0:b1]), _ptr(pe), _ptr(pc), nk,
                                                         out.data_ptr(), nb, N, Nc, ws, nbytes, self.precision, _stream())
                    _lib.check(rc, "fc_flow_log_prob_draws")
                    if nb != B:
                        draws[k0:k1, b0:b1].copy_(out)
            iw = torch.empty((B, N), dtype=torch.float32, device=self.device)
            _lib.check(self.lib.fc_logmeanexp(draws.data_ptr(), K, B * N, iw.data_ptr(), _stream()), "fc_logmeanexp")
        return (iw, draws) if return_draws else iw

    def _ensure_grad(self):
        bad = packing.grad_unsupported_transform(self.config)
        if bad is not None:
            raise _lib.FlowCompareError(f"log_prob_grad: input gradients through {bad} are not supported (affine couplings only)")
        if self._grad is None:
            header, table, arena = packing.pack_flow_grad(self._flow_sd_for_inverse, self.config)
            with torch.cuda.device(self.device):
                arena_dev = arena.to(self.device)
                rc = self.lib.fc_flow_set_grad(self._flow["handle"], header.ctypes.data, len(header), table.ctypes.data, len(table),
                                               arena_dev.data_ptr(), arena_dev.numel())
            _lib.check(rc, "fc_flow_set_grad")
            self._grad = {"arena": arena_dev, "header": header, "table": table}

    def log_prob_grad(self, x, context, extra_context=None, eps=None, workspace_budget=None):
        """Input gradients: (log_prob [B,N], grad [B,N,input_dim]) with grad[b,n] = d log_prob[b,n] / d x[b,n,:input_dim] -- what
        `torch.autograd.grad(flow.log_prob(x, context=...).sum(), x)` gives on the reference (models/transform.py:70-76) with the
        augmentation noise eps held fixed.  A point's log-prob depends on that point and the context only, so this per-point block
        is the whole Jacobian: the gradient of sum(w * log_prob) is w[..., None] * grad.  The context, the extra context and the
        weights are constants.  Arguments as `log_prob`; log_prob is bitwise `log_prob(x, context, eps=eps)`.
        Clouds run in passes of at most 2^16 points (fewer when a pass's workspace would exceed `workspace_budget` bytes); the
        result does not depend on the split.  Affine-coupling flows only: spline / exponential couplings and CIF blocks raise."""
        self._ensure_grad()
        with torch.cuda.device(self.device):
            x, context, Nc, extra, eps, _ = self._flow_inputs("log_prob_grad", x, context, extra_context, eps, None)
            B, N = x.shape[0], x.shape[1]
            if N > GRAD_MAX_PASS_ROWS:
                raise _lib.FlowCompareError(f"log_prob_grad: {N} points per cloud exceed one pass of {GRAD_MAX_PASS_ROWS} rows")
            h = self._flow["handle"]
            wsb = lambda bc: self.lib.fc_flow_log_prob_grad_workspace_bytes(h, bc, N, Nc)
            bc = min(B, GRAD_MAX_PASS_ROWS // N)                              # clouds per pass
            if workspace_budget is not None:
                while bc > 1 and wsb(bc) > workspace_budget:
                    bc = (bc + 1) // 2
            lp = torch.empty((B, N), dtype=torch.float32, device=self.device)
            grad = torch.empty((B, N, self.d_in), dtype=torch.float32, device=self.device)
            for b0 in range(0, B, bc):
                b1 = min(B, b0 + bc)
                nb = b1 - b0
                nbytes = wsb(nb)
                ws = self._workspace(nbytes)
                rc = self.lib.fc_flow_log_prob_grad(h, x[b0:b1].data_ptr(), context[b0:b1].data_ptr(),
                                                    _ptr(None if extra is None else extra[b0:b1]),
                                                    _ptr(None if eps is None else eps[b0:b1]),
                                                    lp[b0:b1].data_ptr(), grad[b0:b1].data_ptr(), nb, N, Nc, ws, nbytes,
                                                    self.precision, _stream())
                _lib.check(rc, "fc_flow_log_prob_grad")
        return lp, grad

    def _prep_context(self, context, extra_context, B):
        context = context.to(self.device)
        if self.is_global and context.dim() == 3:
            context = context[:, 0, :]
        context = _f32c(context, self.device)
        Nc = 1 if self.is_global else context.shape[1]
        extra = None
        if self.has_extra:
            if extra_context is None:
                raise _lib.FlowCompareError("this config uses extra context (extra_z_value_context) but none was given")
            extra = extra_context.to(self.device)
            if extra.dim() == 3:
                extra = extra[:, 0, :]
            extra = _f32c(extra.reshape(B), self.device)
        return context, Nc, extra

    def _eps_cif(self, what, eps_cif, B, N):
        """The CIF blocks' draws [L, B, N, cif_latent_dim - latent_dim] as given (checked) or drawn; None without CIF blocks."""
        if not self.cif_S:
            return None
        eps_cif = self.draw_eps_cif(B, N) if eps_cif is None else _f32c(eps_cif, self.device)
        _check_shape(what, "eps_cif", eps_cif, (self.L, B, N, self.cif_S))
        return eps_cif

    def _flow_inputs(self, what, x, context, extra_context, eps, eps_cif):
        """What a flow pass over x [B, N, >=input_dim] reads: (x cut to input_dim, context, Nc, extra context, eps, eps_cif).
        Noise not given is drawn on the device; given noise of the wrong shape raises.  eps is None for an identity augmenter,
        eps_cif None for a flow without CIF blocks (a given one is then ignored)."""
        x = _f32c(x[..., :self.d_in], self.device)
        B, N = x.shape[0], x.shape[1]
        context, Nc, extra = self._prep_context(context, extra_context, B)
        eps = self.draw_eps(B, N) if eps is None else _f32c(eps, self.device)
        _check_shape(what, "eps", eps, (B, N, self.D - self.d_in))
        return x, context, Nc, extra, eps if self.D > self.d_in else None, self._eps_cif(what, eps_cif, B, N)

    def forward(self, x, context, extra_context=None, eps=None):
        """The forward pass with its latent: returns (log_prob [B,N], z [B,N,latent]) -- `Flow.log_prob` plus the point at
        which the base density was evaluated (what `Flow.sample` inverts)."""
        with torch.cuda.device(self.device):
            x, context, Nc, extra, eps, _ = self._flow_inputs("forward", x, context, extra_context, eps, None)
            B, N = x.shape[0], x.shape[1]
            out = torch.empty((B, N), dtype=torch.float32, device=self.device)
            z = torch.empty((B, N, self.D), dtype=torch.float32, device=self.device)
            nbytes = self.lib.fc_flow_workspace_bytes(self._flow["handle"], B, N, Nc)
            ws = self._workspace(nbytes)
            rc = self.lib.fc_flow_forward(self._flow["handle"], x.data_ptr(), context.data_ptr(), _ptr(extra), _ptr(eps),
                                          out.data_ptr(), z.data_ptr(), B, N, Nc, ws, nbytes, self.precision, _stream())
            _lib.check(rc, "fc_flow_forward")
        return out, z

    @property
    def attention_layer_names(self):
        """Module names (the reference's, e.g. 'transforms.0.attn', 'transforms.1.pre_conditioner.attn') of the attention
        blocks whose weights `attention_maps` returns, in transform order; empty for global-embedding configs."""
        return packing.attention_block_names(self.config)

    def attention_maps(self, x, context, extra_context=None, layers=None, queries=None, eps=None, eps_cif=None):
        """The conditioners' cross-attention weights softmax(q k^T / 8) (reference models/perceiver.py:108-115) from the forward
        pass `log_prob` runs -- what the reference's attention visualisation shows: which context points a target point's
        conditioner attends to, layer by layer.

        Arguments as `log_prob` (`context` is the embedding: `engine.embed(extract_0)`); `layers`: names from
        `attention_layer_names` (None: all); `queries`: indices into the N points of x, any order, repeats allowed (None: all).
        Returns (log_prob [B,N], {name: weights [B, n_query, Nc]}); log_prob is bitwise what `log_prob` returns with the same
        eps, and the maps are views of one allocation."""
        slots, first_slot = self._attention_slots("attention_maps", layers)
        names = self.attention_layer_names
        with torch.cuda.device(self.device):
            B, N = x.shape[0], x.shape[1]
            qidx, n_query = self._query_index("attention_maps", queries, N)
            x, context, Nc, extra, eps, eps_cif = self._flow_inputs("attention_maps", x, context, extra_context, eps, eps_cif)
            slots_host = np.asarray(slots, dtype=np.int32)
            maps = torch.empty((len(slots), B, n_query, Nc), dtype=torch.float32, device=self.device)
            out = torch.empty((B, N), dtype=torch.float32, device=self.device)
            nbytes = self.lib.fc_flow_workspace_bytes(self._flow["handle"], B, N, Nc)
            ws = self._workspace(nbytes)
            rc = self.lib.fc_flow_attention_maps(self._flow["handle"], x.data_ptr(), context.data_ptr(), _ptr(extra), _ptr(eps),
                                                 _ptr(eps_cif), slots_host.ctypes.data, len(slots), _ptr(qidx), n_query,
                                                 maps.data_ptr(), out.data_ptr(), B, N, Nc, ws, nbytes, self.precision, _stream())
            _lib.check(rc, "fc_flow_attention_maps")
        return out, {names[s - first_slot]: maps[i] for i, s in enumerate(slots)}

    def _attention_slots(self, what, layers):
        """(sorted device slots of the named attention blocks, slot of attention_layer_names[0]); raises for global-embedding
        configs, unknown names and an empty list."""
        if self.is_global:
            raise _lib.FlowCompareError(f"{what}: global-embedding configs attend to no context points")
        names = self.attention_layer_names
        first_slot = 0 if self.D > self.d_in else 1      # slot 0 is the augmenter's attention (absent for an identity augmenter)
        if layers is None:
            layers = names
        unknown = [n for n in layers if n not in names]
        if unknown or not layers:
            raise _lib.FlowCompareError(f"{what}: unknown layer names {unknown}; choose from attention_layer_names"
                                        if unknown else f"{what}: no layers requested")
        return sorted({names.index(n) + first_slot for n in layers}), first_slot

    def _query_index(self, what, queries, N):
        """(device int32 query rows or None for all, n_query) from indices into the N points of a cloud."""
        if queries is None:
            return None, N
        q = torch.as_tensor(queries).reshape(-1)
        if q.numel() == 0 or q.is_floating_point() or int(q.min()) < 0 or int(q.max()) >= N:
            raise _lib.FlowCompareError(f"{what}: query indices must be integers in [0, {N})")
        qidx = q.to(device=self.device, dtype=torch.int32).contiguous()
        return qidx, qidx.numel()

    def attention_score_grads(self, x, context, extra_context=None, layers=None, queries=None, eps=None, sum_layers=False,
                              workspace_budget=None):
        """Attention score gradients: d log_prob[b, i] / d s_ij for the attention scores s = q k^T / 8 of chosen blocks (reference
        models/perceiver.py:108-115) -- what `sim.grad` holds on the reference after `sim.retain_grad()` and
        `flow.log_prob(x, context=...).sum().backward()`, with the augmentation noise eps held fixed.  The signed answer to which
        context points raise (positive) or lower (negative) a target point's likelihood if its conditioner attended to them more;
        a row sums to zero.  Formed from the input-gradient pass `log_prob_grad` runs; no gradient flows to the context.

        Arguments as `attention_maps` (`layers` from `attention_layer_names`, None: all; `queries` any order, repeats allowed)
        and `log_prob_grad` (passes of at most 2^16 points, fewer under `workspace_budget`; the result does not depend on the
        split).  Returns (log_prob [B,N], grad [B,N,input_dim], maps): log_prob and grad bitwise `log_prob_grad`'s, maps
        {name: [B, n_query, Nc]}, or with `sum_layers` one [B, n_query, Nc] tensor, the sum over the selected blocks (the
        gradient with respect to a logit bias they all share; one block's memory for any number of blocks), added in fp32 in the
        order of the backward walk: the last coupling layer's block first, the augmenter's last.  Affine-coupling flows only."""
        slots, first_slot = self._attention_slots("attention_score_grads", layers)
        names = self.attention_layer_names
        with torch.cuda.device(self.device):
            B, N = x.shape[0], x.shape[1]
            qidx, n_query = self._query_index("attention_score_grads", queries, N)
            self._ensure_grad()
            x, context, Nc, extra, eps, _ = self._flow_inputs("attention_score_grads", x, context, extra_context, eps, None)
            if N > GRAD_MAX_PASS_ROWS:
                raise _lib.FlowCompareError(f"attention_score_grads: {N} points per cloud exceed one pass of {GRAD_MAX_PASS_ROWS} rows")
            h = self._flow["handle"]
            wsb = lambda bc: self.lib.fc_flow_log_prob_grad_workspace_bytes(h, bc, N, Nc)
            bc = min(B, GRAD_MAX_PASS_ROWS // N)                              # clouds per pass
            if workspace_budget is not None:
                while bc > 1 and wsb(bc) > workspace_budget:
                    bc = (bc + 1) // 2
            slots_host = np.asarray(slots, dtype=np.int32)
            lp = torch.empty((B, N), dtype=torch.float32, device=self.device)
            grad = torch.empty((B, N, self.d_in), dtype=torch.float32, device=self.device)
            shape = (B, n_query, Nc) if sum_layers else (len(slots), B, n_query, Nc)
            maps = torch.empty(shape, dtype=torch.float32, device=self.device)
            for b0 in range(0, B, bc):
                b1 = min(B, b0 + bc)
                nb = b1 - b0
                dst = maps[b0:b1] if sum_layers else maps[:, b0:b1]
                out = dst if dst.is_contiguous() else torch.empty(dst.shape, dtype=torch.float32, device=self.device)
                nbytes = wsb(nb)
                ws = self._workspace(nbytes)
                rc = self.lib.fc_flow_attention_score_grads(h, x[b0:b1].data_ptr(), context[b0:b1].data_ptr(),
                                                            _ptr(None if extra is None else extra[b0:b1]),
                                                            _ptr(None if eps is None else eps[b0:b1]), slots_host.ctypes.data,
                                                            len(slots), _ptr(qidx), n_query, 1 if sum_layers else 0,
                                                            out.data_ptr(), lp[b0:b1].data_ptr(), grad[b0:b1].data_ptr(), nb, N,
                                                            Nc, ws, nbytes, self.precision, _stream())
                _lib.check(rc, "fc_flow_attention_score_grads")
                if out is not dst:
                    dst.copy_(out)
        if sum_layers:
            return lp, grad, maps
        return lp, grad, {names[s - first_slot]: maps[i] for i, s in enumerate(slots)}

    # ------------------------------------------------------------------ inverse / sampling pass
    def _ensure_inverse(self):
        if self._inv is None:
            header, table, arena = packing.pack_flow_inverse(self._flow_sd_for_inverse, self.config, self._tc_format)
            with torch.cuda.device(self.device):
                arena_dev = arena.to(self.device)
                rc = self.lib.fc_flow_set_inverse(self._flow["handle"], header.ctypes.data, len(header), table.ctypes.data, len(table),
                                                  arena_dev.data_ptr(), arena_dev.numel())
            _lib.check(rc, "fc_flow_set_inverse")
            self._inv = {"arena": arena_dev, "header": header, "table": table}

    def sample(self, n_points, context, extra_context=None, z=None, seed=None, eps_cif=None):
        """`Flow.sample(num_samples=1, n_points=, context=, extra_context=)` (reference models/transform.py:79-84):
        z ~ sample_dist = N(loc, scale) [B, n_points, latent] (or the injected `z`), then every transform's inverse.
        eps_cif [L, B, n_points, cif_latent_dim - latent_dim]: the CIF blocks' `Slice.inverse` draws (default: drawn on the device).
        Returns x [B, n_points, input_dim]."""
        self._ensure_inverse()
        with torch.cuda.device(self.device):
            B = context.shape[0]
            context, Nc, extra = self._prep_context(context, extra_context, B)
            if z is None:
                z = torch.empty((B, n_points, self.D), dtype=torch.float32, device=self.device)
                if seed is None:
                    seed = self._next_seed()
                _lib.check(self.lib.fc_fill_normal(z.data_ptr(), z.numel(), seed, 0, _stream()), "fc_fill_normal")
                z = z * self._sample_scale + self._sample_loc
            z = _f32c(z, self.device).reshape(B, n_points, self.D)
            out = torch.empty((B, n_points, self.d_in), dtype=torch.float32, device=self.device)
            nbytes = self.lib.fc_flow_workspace_bytes(self._flow["handle"], B, n_points, Nc)
            ws = self._workspace(nbytes)
            eps_cif = self._eps_cif("sample", eps_cif, B, n_points)
            if self.cif_S:
                rc = self.lib.fc_flow_sample_cif(self._flow["handle"], z.data_ptr(), context.data_ptr(), _ptr(extra),
                                                 eps_cif.data_ptr(), out.data_ptr(), B, n_points, Nc, ws, nbytes, self.precision,
                                                 _stream())
                _lib.check(rc, "fc_flow_sample_cif")
            else:
                rc = self.lib.fc_flow_sample(self._flow["handle"], z.data_ptr(), context.data_ptr(), _ptr(extra), out.data_ptr(), B,
                                             n_points, Nc, ws, nbytes, self.precision, _stream())
                _lib.check(rc, "fc_flow_sample")
        return out

    def make_sample(self, n_points, extract_0, extra_context=None, z=None, seed=None, eps_cif=None):
        """`make_sample(n_points, extract_0, models_dict, config, sample_distrib=None, extra_context=None)` (reference
        model_initialization.py:231-245): embed the context cloud, then the generative pass.  Returns what the reference
        returns: x [B, n_points, input_dim] with singleton dimensions squeezed."""
        emb = self.embed(extract_0)
        return self.sample(n_points, emb, extra_context=extra_context, z=z, seed=seed, eps_cif=eps_cif).squeeze()

    # ------------------------------------------------------------------ whole path
    def inner_loop(self, batch, eps=None, eps_cif=None):
        """`inner_loop(batch, models_dict, config)` (reference model_initialization.py:206-228).
        batch = (extract_0 [B,Nc,>=6], extract_1 [B,N,>=6], extra_context [B,1] | None).
        Returns (loss, log_prob [B,N], bpd) as CUDA tensors."""
        e0, e1, extra = batch
        if self.cif_S or self.D == self.d_in:
            # flows outside the shipped architectures (CIF blocks / identity augmenter): embed, then the flow, as two calls
            lp = self.log_prob(e1, self.embed(e0), extra_context=extra, eps=eps, eps_cif=eps_cif)
            loss = -lp.mean()
            return loss, lp, loss * math.log2(math.e) / self.d_in
        with torch.cuda.device(self.device):
            e0 = _f32c(e0[:, :, :self.d_in], self.device)
            e1 = _f32c(e1[:, :, :self.d_in], self.device)
            B, Nc, N = e0.shape[0], e0.shape[1], e1.shape[1]
            ex = None
            if self.has_extra:
                if extra is None:
                    raise _lib.FlowCompareError("this config uses extra context but batch[2] is None")
                ex = _f32c(extra.reshape(B), self.device)
            eps = self.draw_eps(B, N) if eps is None else _f32c(eps, self.device)
            lp = torch.empty((B, N), dtype=torch.float32, device=self.device)
            stats = torch.empty(2, dtype=torch.float32, device=self.device)
            nbytes = self.lib.fc_inner_loop_workspace_bytes(self._emb["handle"], self._flow["handle"], B, N, Nc)
            ws = self._workspace(nbytes)
            rc = self.lib.fc_inner_loop(self._emb["handle"], self._flow["handle"], e0.data_ptr(), e1.data_ptr(), _ptr(ex),
                                        eps.data_ptr(), lp.data_ptr(), stats.data_ptr(), B, N, Nc, ws, nbytes,
                                        self.precision, _stream())
            _lib.check(rc, "fc_inner_loop")
        return stats[0], lp, stats[1]

    def capture_inner_loop(self, B, Nc, N):
        """CUDA-graph version of `inner_loop` for a fixed (B, Nc, N): the ~40 kernel launches per flow layer (4.6 k per
        forward at 115 layers) are captured once and replayed with one launch, which is what matters at small batch sizes
        where the forward is launch bound (B = 1: ~25 ms of launches for ~10 ms of kernels).  Returns a callable
        `run(e0, e1, extra, eps=None) -> (loss, log_prob, bpd)`; inputs are copied into the graph's static buffers, results
        are views of static buffers (clone them to keep them across calls)."""
        dev = self.device
        with torch.cuda.device(dev):
            st = {"e0": torch.zeros(B, Nc, self.d_in, device=dev), "e1": torch.zeros(B, N, self.d_in, device=dev),
                  "extra": torch.zeros(B, device=dev) if self.has_extra else None,
                  "eps": torch.zeros(B, N, self.D - self.d_in, device=dev)}
            saved_ws, self._ws = self._ws, None     # the graph gets its OWN workspace (the shared one may be re-allocated later)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):          # warm-up outside capture: lazy attribute / tensor-map / workspace setup
                for _ in range(2):
                    out = self.inner_loop((st["e0"], st["e1"], st["extra"]), eps=st["eps"])
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self.inner_loop((st["e0"], st["e1"], st["extra"]), eps=st["eps"])
            graph_ws, self._ws = self._ws, saved_ws
        engine = self

        def run(e0, e1, extra=None, eps=None, copy=True):
            if copy:
                st["e0"].copy_(e0[:, :, :engine.d_in])
                st["e1"].copy_(e1[:, :, :engine.d_in])
                if st["extra"] is not None:
                    st["extra"].copy_(extra.reshape(B))
                if eps is None:
                    st["eps"].copy_(engine.draw_eps(B, N))
                else:
                    st["eps"].copy_(eps)
            g.replay()
            return out
        run.graph, run.static, run.workspace = g, st, graph_ws
        return run

    def inner_loop_host(self, e0, e1, extra, eps, out_log_prob=None, out_stats=None):
        """Same path through `fc_inner_loop_host`: HOST (ideally pinned) fp32 contiguous buffers in and out,
        copies on the current stream, synchronous on return.  Used by the end-to-end benchmark."""
        for t in (e0, e1, eps) + ((extra,) if extra is not None else ()):
            assert t.device.type == "cpu" and t.dtype == torch.float32 and t.is_contiguous()
        assert e0.shape[2] == self.d_in and e1.shape[2] == self.d_in
        B, Nc, N = e0.shape[0], e0.shape[1], e1.shape[1]
        if out_log_prob is None:
            out_log_prob = torch.empty((B, N), dtype=torch.float32).pin_memory()
        if out_stats is None:
            out_stats = torch.empty(2, dtype=torch.float32).pin_memory()
        with torch.cuda.device(self.device):
            nbytes = self.lib.fc_inner_loop_host_workspace_bytes(self._emb["handle"], self._flow["handle"], B, N, Nc)
            ws = self._workspace(nbytes)
            rc = self.lib.fc_inner_loop_host(self._emb["handle"], self._flow["handle"], e0.data_ptr(), e1.data_ptr(),
                                             _ptr(extra), eps.data_ptr(), out_log_prob.data_ptr(), out_stats.data_ptr(),
                                             B, N, Nc, ws, nbytes, self.precision, _stream())
            _lib.check(rc, "fc_inner_loop_host")
        return out_stats[0], out_log_prob, out_stats[1]

    # ------------------------------------------------------------------ consumers
    def change_maps(self, batch_1_0, batch_0_0, batch_0_1, batch_1_1, multiple=3.0, hard_cutoff=None, eps=None, n_draws=1):
        """The four `inner_loop` passes + two `log_prob_to_change` calls of `DatasetViewer.view_index`
        (reference test_flow.py:39-62) as ONE batched pass: the four batches (1|0, 0|0, 0|1, 1|1; each
        (extract_0, extract_1, extra_context)) are stacked along the batch axis -- cloud pairs are independent and a
        pair's result does not depend on what else is in the batch (tested bitwise) -- and the change scores are then
        formed per direction exactly as the reference does.  eps: optional [4B, N, latent-input_dim] noise.
        Returns a dict of CUDA tensors: log_prob_{1_0,0_0,0_1,1_1} [B,N], change_1_0, change_0_1 [B,N], loss_{1_0,...}
        (= -mean log_prob, `inner_loop`'s first return) and nats_{1_0,...} (= loss * log2(e) / input_dim, its third return, which
        the reference's evaluation prints as "nats", test_flow.py:160,224).
        n_draws > 1: every log_prob is `log_prob_iw` over that many augmentation draws (the same stacked batches; eps
        [n_draws, 4B, N, latent-input_dim]), so the change masks and loss / nats are those of the importance-weighted estimate.
        n_draws = 1 is the reference's single-draw estimator and runs the path above unchanged."""
        K = _n_draws(n_draws, "change_maps")
        batches = (batch_1_0, batch_0_0, batch_0_1, batch_1_1)
        B = batches[0][0].shape[0]
        for b in batches:
            if b[0].shape[0] != B or b[0].shape[1] != batches[0][0].shape[1] or b[1].shape[1] != batches[0][1].shape[1]:
                raise _lib.FlowCompareError("change_maps: the four batches must have the same batch size and cloud sizes")
        e0 = torch.cat([b[0][:, :, :self.d_in].to(self.device, torch.float32) for b in batches], dim=0)
        e1 = torch.cat([b[1][:, :, :self.d_in].to(self.device, torch.float32) for b in batches], dim=0)
        extra = None
        if self.has_extra:
            if any(b[2] is None for b in batches):
                raise _lib.FlowCompareError("this config uses extra context but a batch has none")
            extra = torch.cat([b[2].reshape(B).to(self.device, torch.float32) for b in batches], dim=0)
        # context clouds that are the SAME tensor in several batches (a caller that normalised them once) are embedded once
        uniq, slot = [], []
        for b in batches:
            for j, u in enumerate(uniq):
                if u is b[0]:
                    slot.append(j)
                    break
            else:
                slot.append(len(uniq))
                uniq.append(b[0])
        if K > 1 or (len(uniq) < 4 and not self.cif_S and self.D > self.d_in):
            emb = self.embed(torch.cat([u[:, :, :self.d_in].to(self.device, torch.float32) for u in uniq], dim=0))
            ctx = torch.cat([emb[j * B:(j + 1) * B] for j in slot], dim=0)
            if K > 1:
                lp = self.log_prob_iw(e1, ctx, extra_context=extra, n_draws=K, eps=eps)
            else:
                lp = self.log_prob(e1, ctx, extra_context=extra, eps=eps)
        else:
            _, lp, _ = self.inner_loop((e0, e1, extra), eps=eps)
        names = ("1_0", "0_0", "0_1", "1_1")
        out = {}
        for i, nm in enumerate(names):
            out["log_prob_" + nm] = lp[i * B:(i + 1) * B]
            out["loss_" + nm] = -out["log_prob_" + nm].mean()                                   # inner_loop's first return
            out["nats_" + nm] = out["loss_" + nm] * math.log2(math.e) / self.d_in               # its third: what test_flow.py:160,224 call "nats"
        out["change_1_0"] = log_prob_to_change(out["log_prob_1_0"], out["log_prob_0_0"], multiple, hard_cutoff)
        out["change_0_1"] = log_prob_to_change(out["log_prob_0_1"], out["log_prob_1_1"], multiple, hard_cutoff)
        return out

    def evaluate_on_batches(self, batches, multiple=5.4, hard_cutoff=None, eps=None, n_draws=1):
        """The evaluation loop of `evaluate_on_test` (reference test_flow.py:147-226) over an iterable of
        `(batch_1_0, batch_0_0)` pairs, each batch `(extract_0, extract_1, extra_context)` as the reference assembles them
        (test_flow.py:155-158): the two passes run as ONE stacked pass, then `log_prob_to_change(lp_1_0, lp_0_0, multiple)`,
        the per-cloud change means `(change > 0).float().mean(-1)` (:172) and the running average of the 1|0 pass's nats
        (:224-226).  eps: optional iterable of [2B, N, latent-input_dim] noise per batch (1|0 rows first).
        Returns `(nats_avg, change_mean_list)` as Python floats, like the reference.
        n_draws > 1: the log-probs are `log_prob_iw` over that many augmentation draws (eps per batch [n_draws, 2B, N,
        latent-input_dim]), so the change means and nats are those of the importance-weighted estimate; n_draws = 1 is the
        reference's single-draw estimator and runs the path above unchanged."""
        K = _n_draws(n_draws, "evaluate_on_batches")
        nats_avg, change_mean_list = 0.0, []
        eps_it = iter(eps) if eps is not None else None
        for batch_ind, (b10, b00) in enumerate(batches):
            B = b10[0].shape[0]
            e0 = torch.cat([b[0][:, :, :self.d_in].to(self.device, torch.float32) for b in (b10, b00)], dim=0)
            e1 = torch.cat([b[1][:, :, :self.d_in].to(self.device, torch.float32) for b in (b10, b00)], dim=0)
            extra = None
            if self.has_extra:
                if b10[2] is None or b00[2] is None:
                    raise _lib.FlowCompareError("this config uses extra context but a batch has none")
                extra = torch.cat([b[2].reshape(-1).to(self.device, torch.float32) for b in (b10, b00)], dim=0)
            eps_b = None if eps_it is None else next(eps_it)
            if K > 1:
                lp = self.log_prob_iw(e1, self.embed(e0), extra_context=extra, n_draws=K, eps=eps_b)
            else:
                _, lp, _ = self.inner_loop((e0, e1, extra), eps=eps_b)
            lp10, lp00 = lp[:B], lp[B:]
            change = log_prob_to_change(lp10, lp00, multiple, hard_cutoff)
            change_mean_list.extend((change > 0).float().mean(dim=-1).tolist())
            nats = (-lp10.mean() * math.log2(math.e) / self.d_in).item()
            nats_avg = (nats_avg * batch_ind + nats) / (batch_ind + 1)
        return nats_avg, change_mean_list

    def log_prob_to_change(self, log_prob_1_given_0, log_prob_0_given_0, multiple, hard_cutoff=None):
        """`log_prob_to_change` (+ `clamp_infs`), reference test_flow.py:241-275."""
        return log_prob_to_change(log_prob_1_given_0, log_prob_0_given_0, multiple, hard_cutoff)


# ---------------------------------------------------------------------- free functions (op level)
def knn(x, k):
    """`knn(x, k)` of reference models/pytorch_gcn.py:13-20: x [B,C,N] CUDA -> idx [B,N,k] int64."""
    lib = _lib.load()
    assert x.is_cuda
    pts = x.transpose(2, 1).to(torch.float32).contiguous()  # [B,N,C]
    B, N, C = pts.shape
    idx = torch.empty((B, N, k), dtype=torch.int64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.fc_knn_self(pts.data_ptr(), C, B, N, C, k, 0, idx.data_ptr(), _stream()), "fc_knn_self")
    return idx


def get_knn(samples, context_cloud, n_neighbors):
    """`get_knn(samples, context_cloud, n_neighbors)` of reference knn.py:79-90 ('torch' flavour):
    [Nq,D], [Nt,D] CUDA -> [Nq,k] int64, ascending distance."""
    lib = _lib.load()
    assert samples.is_cuda and context_cloud.is_cuda
    q = samples.to(torch.float32).contiguous()
    t = context_cloud.to(torch.float32).contiguous()
    idx = torch.empty((q.shape[0], n_neighbors), dtype=torch.int64, device=q.device)
    with torch.cuda.device(q.device):
        _lib.check(lib.fc_knn_query(q.data_ptr(), t.data_ptr(), q.shape[0], t.shape[0], q.shape[1], n_neighbors,
                                    idx.data_ptr(), _stream()), "fc_knn_query")
    return idx


def log_prob_to_change(log_prob_1_given_0, log_prob_0_given_0, multiple, hard_cutoff=None):
    """`log_prob_to_change` of reference test_flow.py:249-275 on CUDA tensors [B,N] (or [N])."""
    lib = _lib.load()
    a, c = log_prob_1_given_0, log_prob_0_given_0
    assert a.is_cuda and c.is_cuda
    squeeze = a.dim() == 1
    a2 = a.reshape(-1, a.shape[-1]).to(torch.float32).contiguous()
    c2 = c.reshape(-1, c.shape[-1]).to(torch.float32).contiguous()
    out = torch.empty_like(a2)
    with torch.cuda.device(a.device):
        _lib.check(lib.fc_change_score(a2.data_ptr(), c2.data_ptr(), out.data_ptr(), a2.shape[0], a2.shape[1],
                                       float(multiple), 0 if hard_cutoff is None else 1,
                                       0.0 if hard_cutoff is None else float(hard_cutoff), _stream()), "fc_change_score")
    return out[0] if squeeze else out.reshape(a.shape)


# ---------------------------------------------------------------------- drop-in adapters
class _LogProbFunction(torch.autograd.Function):
    """log_prob(x | context) with a backward for x: the forward is the plain `log_prob` with an explicit eps (so a caller that never
    calls backward pays nothing extra), the backward `log_prob_grad` with that eps.  Context and extra context are constants."""

    @staticmethod
    def forward(ctx, x, context, extra_context, engine, eps):
        ctx.engine, ctx.context, ctx.extra = engine, context, extra_context
        ctx.save_for_backward(x, eps)
        return engine.log_prob(x, context, extra_context, eps=eps)

    @staticmethod
    def backward(ctx, grad_output):
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            raise _lib.FlowCompareError("log_prob backward: gradients with respect to the context or the extra context are not "
                                        "supported (only the target points x)")
        x, eps = ctx.saved_tensors
        _, g = ctx.engine.log_prob_grad(x.detach(), ctx.context, ctx.extra, eps=eps)
        g = grad_output.to(g.device, g.dtype)[..., None] * g
        if x.shape[-1] > g.shape[-1]:       # columns past input_dim do not enter the flow
            g = torch.cat((g, g.new_zeros(g.shape[:-1] + (x.shape[-1] - g.shape[-1],))), dim=-1)
        return g.to(x.device, x.dtype), None, None, None, None


class _FlowAdapter:
    """Stands in for `models.Flow` inside a models_dict: same `log_prob` signature."""

    def __init__(self, engine):
        self.engine = engine
        self.eps = None  # set to a tensor to inject the augmentation noise (parity tests)
        self.z = None    # set to a tensor to inject the base draw of `sample` (parity tests)

    def log_prob(self, x, context=None, extra_context=None):
        """`Flow.log_prob`.  With grad mode on and `x.requires_grad`, the result is differentiable with respect to x (the reference's
        autograd through the flow, eps held at the value this call drew): backward runs `log_prob_grad`.  Otherwise this is the
        plain call."""
        if torch.is_grad_enabled() and isinstance(x, torch.Tensor) and x.requires_grad:
            eps = self.eps if self.eps is not None else self.engine.draw_eps(x.shape[0], x.shape[1])
            return _LogProbFunction.apply(x, context, extra_context, self.engine, eps)
        return self.engine.log_prob(x, context, extra_context, eps=self.eps)

    def sample(self, num_samples, n_points, context=None, sample_distrib=None, extra_context=None):
        """`Flow.sample` (models/transform.py:79-84); `sample_distrib` may be any object with the reference's
        `.sample(num_samples, n_points=)` (it is asked for the base draw exactly as the reference asks it)."""
        z = None
        if sample_distrib is not None:
            z = sample_distrib.sample(num_samples, n_points=n_points)
        elif self.z is not None:
            z = self.z
        assert num_samples == 1, "the reference only ever draws num_samples=1 (model_initialization.py:243)"
        return self.engine.sample(n_points, context, extra_context=extra_context, z=z)

    def eval(self):
        return self


class _EmbedderAdapter:
    def __init__(self, engine):
        self.engine = engine

    def __call__(self, extract_0):
        return self.engine.embed(extract_0)

    def eval(self):
        return self


def accelerate(models_dict, config, device="cuda:0", precision="fp32"):
    """Returns a models_dict the reference's own `inner_loop(batch, models_dict, config)` accepts
    (model_initialization.py:206-228), backed by the CUDA path."""
    engine = FlowCompareB200(models_dict, config, device=device, precision=precision)
    return {"parameters": models_dict.get("parameters", []), "flow": _FlowAdapter(engine),
            "input_embedder": _EmbedderAdapter(engine), "engine": engine}


def inner_loop(batch, models_dict, config, eps=None):
    """Same signature as the reference's `inner_loop`; `models_dict` must come from `accelerate`."""
    return models_dict["engine"].inner_loop(batch, eps=eps)


def make_sample(n_points, extract_0, models_dict, config, sample_distrib=None, extra_context=None):
    """Same signature as the reference's `make_sample` (model_initialization.py:231-245); `models_dict` from `accelerate`."""
    eng = models_dict["engine"]
    z = None if sample_distrib is None else sample_distrib.sample(1, n_points=n_points)
    return eng.make_sample(n_points, extract_0, extra_context=extra_context, z=z)
