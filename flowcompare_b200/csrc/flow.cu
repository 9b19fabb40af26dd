// The conditional normalizing flow: `Flow.log_prob` of reference models/transform.py:70-76 over the
// transform list of model_initialization.py:134-152, as a stream of fused GEMM / attention launches.
//
// Per coupling layer (attention configs), with M = B*N rows:
//   pre-attention MLP (reference models/cif_block.py:14-20, models/nets.py:19-30)   4 GEMMs (GELU/residual fused)
//   LayerNorm row statistics (models/perceiver.py:26-35)                            1 small kernel
//   to_q with LayerNorm folded into the epilogue (perceiver.py:109)                 1 GEMM
//   to_kv on the context (perceiver.py:110)                                         1 GEMM
//   softmax(q k^T / 8) v, flash style (perceiver.py:111-113)                        1 kernel
//   coupling MLP; attention out-projection (perceiver.py:95-96) and the concat with x1 / extra
//   context (transform.py:49-50, affine_coupling.py:34-35) folded into its first layer           4 GEMMs
//     last GEMM's epilogue = sigmoid scale, y2 = x2*s + t in place, sum log s -> partial log-det
//   ActNorm + LinearLU folded into one 300x300 GEMM (act_norm.py:37-43, permuters.py:164-169)     1 GEMM
// The running log-det never leaves fp32 registers/partials until the final reduction.
#include "model.cuh"
#include <new>

namespace {

__global__ void copy_cols_kernel(const float* __restrict__ src, int lds, float* __restrict__ dst, int ldd,
                                 long long M, int cols) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * cols) return;
    const long long r = i / cols; const int c = (int)(i % cols);
    dst[r * ldd + c] = src[r * lds + c];
}

// one warp per row: mean and 1/sqrt(var + eps) (biased variance, two passes in registers).  VEC: 16-byte loads
// (width % 4 == 0, 16-byte aligned rows) -- the scalar form reached only ~1.8 TB/s.
template <bool VEC>
__global__ void ln_stats_kernel(const float* __restrict__ h, int ldh, int M, int width, float eps,
                                float* __restrict__ mu, float* __restrict__ rstd) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= M) return;
    const float* p = h + (size_t)row * ldh;
    float v[16];
    float s = 0.f;
    if (VEC) {
        const float4* p4 = reinterpret_cast<const float4*>(p);
        const int n4 = width >> 2;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = i * 32 + lane;
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < n4) x = __ldg(p4 + c);
            v[4 * i] = x.x; v[4 * i + 1] = x.y; v[4 * i + 2] = x.z; v[4 * i + 3] = x.w;
            s += (x.x + x.y) + (x.z + x.w);
        }
    } else {
        const int per = (width + 31) / 32;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            v[i] = 0.f;
            if (i < per) { const int c = i * 32 + lane; if (c < width) { v[i] = p[c]; s += v[i]; } }
        }
    }
    s = fc_warp_sum(s);
    const float m = s / (float)width;
    float q = 0.f;
    if (VEC) {
        const int n4 = width >> 2;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (i * 32 + lane < n4) {
#pragma unroll
                for (int e = 0; e < 4; ++e) { const float d = v[4 * i + e] - m; q = fmaf(d, d, q); }
            }
    } else {
        const int per = (width + 31) / 32;
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (i < per) { const int c = i * 32 + lane; if (c < width) { const float d = v[i] - m; q = fmaf(d, d, q); } }
    }
    q = fc_warp_sum(q);
    if (lane == 0) { mu[row] = m; rstd[row] = rsqrtf(q / (float)width + eps); }
}

// cbA[b] = [extra_b (if extra) | ctx_b (if global)], zero padded to lda
__global__ void build_cb_input_kernel(const float* __restrict__ extra, const float* __restrict__ ctx, int E,
                                      int has_extra, int is_global, int B, int lda, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * lda) return;
    const int b = i / lda, c = i % lda;
    float v = 0.f;
    if (has_extra && c == 0) v = extra[b];
    else if (is_global) { const int e = c - has_extra; if (e >= 0 && e < E) v = ctx[(size_t)b * E + e]; }
    out[i] = v;
}

// log_prob = sum(augment partials) + sum(coupling partials) + const + sum_d(-0.5 z_d^2 - 0.5 log 2pi)
// (reference models/distributions.py:192-195 for the base density).  One warp per row.  K > 1: rows are in the K-draw
// layout (b*K + k)*N + n and the value goes to log_prob[k][b][n] (draw-major); K == 1: to log_prob[row].
__global__ void finalize_kernel(const float* __restrict__ z, int ldz, int D, const float* __restrict__ apart,
                                int n_apart, const float* __restrict__ cpart, int n_cpart, int M, float ldj_const,
                                float* __restrict__ log_prob, int N, int K) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= M) return;
    const float* p = z + (size_t)row * ldz;
    float s = 0.f;
    for (int c = lane; c < D; c += 32) { const float v = p[c]; s += -0.91893853320467274178f - 0.5f * v * v; }
    s = fc_warp_sum(s);
    if (lane == 0) {
        float acc = 0.f;
        for (int i = 0; i < n_apart; ++i) acc += apart[(size_t)i * M + row];
        for (int i = 0; i < n_cpart; ++i) acc += cpart[(size_t)i * M + row];
        const int out = K == 1 ? row : ((row / N) % K) * (M / K) + (row / (K * N)) * N + row % N;
        log_prob[out] = (acc + ldj_const) + s;
    }
}

}  // namespace

int fc_launch_ln_stats(const float* h, int ldh, int M, int width, float eps, float* mu, float* rstd, cudaStream_t s) {
    FC_REQUIRE(width <= 512);
    const int wpb = 8;
    if ((width & 3) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(h) & 15) == 0)
        ln_stats_kernel<true><<<(M + wpb - 1) / wpb, wpb * 32, 0, s>>>(h, ldh, M, width, eps, mu, rstd);
    else
        ln_stats_kernel<false><<<(M + wpb - 1) / wpb, wpb * 32, 0, s>>>(h, ldh, M, width, eps, mu, rstd);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

static int copy_cols(const float* src, int lds, float* dst, int ldd, long long M, int cols, cudaStream_t s) {
    const long long tot = M * cols;
    copy_cols_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(src, lds, dst, ldd, M, cols);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

// an MLP's first layer on its input [A1 | A2], with the per-cloud bias in place of the packed one when `in` carries one
static GemmArgs mlp_in_gemm(const FcMlp& m, const FcMlpIn& in, float* C, int ldc, int M, int precision) {
    GemmArgs g = fc_gemm_linear(m.in, in.A1, in.lda1, C, ldc, M, precision);
    g.A2 = in.A2; g.lda2 = in.lda2;
    if (in.bias) { g.bias = in.bias; g.bias_ld = in.bias_ld; g.bias_group = in.bias_group; }
    return g;
}

int fc_run_mlp_hidden(const FcMlp& m, const FcMlpIn& in, int M, float* bufA, float* bufB, int ldh, int precision,
                      cudaStream_t stream, float** last) {
    // reference models/nets.py:19-30: x = act(in(x)); even hidden i: res = x, x = act(layer(x));
    // odd i: x = act(res + layer(x))
    GemmArgs g = mlp_in_gemm(m, in, bufA, ldh, M, precision);
    g.act = m.act;
    int rc = fc_launch_gemm(g, stream);
    if (rc) return rc;
    float* cur = bufA; float* other = bufB;
    for (int i = 0; i < m.n_hidden; ++i) {
        g = fc_gemm_linear(m.hidden[i], cur, ldh, other, ldh, M, precision);
        g.act = m.act;
        // odd i: the residual source is `other` (the activation before the previous layer); written in place over it
        if (i & 1) { g.res = other; g.ldres = ldh; }
        rc = fc_launch_gemm(g, stream);
        if (rc) return rc;
        float* t = cur; cur = other; other = t;
    }
    *last = cur;
    return FC_OK;
}

// ------------------------------------------------------------------------------------------ create
static FcAttn read_attn(FcCursor& c, const fc_flow& f) {
    FcAttn a;
    a.csum = c.ptr(c.next(), f.inner);
    a.qbias = c.ptr(c.next(), f.inner);
    a.q = c.linear(f.attn_in, 0, f.inner, /*has_bias=*/false);
    a.kv = c.linear(f.E, 0, 2 * f.inner, /*has_bias=*/false);
    if (!a.csum || !a.qbias) c.ok = false;
    return a;
}

extern "C" int fc_flow_create(const int32_t* header, int n_header, const int64_t* table, int n_table,
                              const float* arena, int64_t arena_floats, fc_flow** out) {
    FC_REQUIRE(header && table && arena && out && n_header >= 19);
    if (header[0] != FC_FLOW_MAGIC || (header[1] != FC_ARENA_VERSION && header[1] != FC_ARENA_VERSION_F16)) return FC_ERR_MODEL;
    if (reinterpret_cast<uintptr_t>(arena) & 15) return FC_ERR_MODEL;
    fc_flow* f = new (std::nothrow) fc_flow();
    if (!f) return FC_ERR_MODEL;
    f->L = header[2]; f->D = header[3]; f->d_in = header[4]; f->half = header[5]; f->extra = header[6];
    f->is_global = header[7]; f->E = header[8]; f->inner = header[9]; f->attn_in = header[10];
    f->hid = header[11]; f->n_hid = header[12]; f->pre_hid = header[13]; f->n_pre_hid = header[14];
    f->aug_hid = header[15]; f->n_aug_hid = header[16]; f->augpre_hid = header[17]; f->n_augpre_hid = header[18];
    f->arena = arena; f->arena_floats = arena_floats;
    if (n_header >= 29) {
        f->cpl_kind = header[19]; f->num_bins = header[20]; f->act = header[21]; f->has_aug = header[22];
        f->cif_dim = header[23]; f->cif_hid = header[24]; f->n_cif_hid = header[25]; f->affcif_hid = header[26];
        f->n_affcif_hid = header[27];
        memcpy(&f->cif_clamp, &header[28], sizeof(float));
    }
    const int n2 = f->D - f->half, S = f->cif_dim ? f->cif_dim - f->D : 0;
    bool dims_ok = f->L >= 1 && f->D >= 2 && f->D <= 512 && f->d_in >= 1 && f->d_in <= f->D && f->half == f->D / 2 &&
                   f->inner == 64 && f->attn_in <= 512 && f->hid <= 512 && f->pre_hid <= 512 && f->aug_hid <= 512 &&
                   f->augpre_hid <= 512 && (f->D % 2) == 0 && ((f->D - f->d_in) % 2) == 0 &&
                   (f->has_aug ? (f->d_in < f->D && f->hid == f->aug_hid) : f->d_in == f->D) &&
                   f->cpl_kind >= FC_CPL_AFFINE && f->cpl_kind <= FC_CPL_EXPO && (f->act == FC_ACT_GELU || f->act == FC_ACT_RELU) &&
                   (f->cpl_kind != FC_CPL_SPLINE || (f->num_bins >= 1 && f->num_bins <= 16)) &&
                   (f->cpl_kind != FC_CPL_EXPO || n2 <= fc_expm_max_n()) &&
                   (f->cif_dim == 0 || (S > 0 && f->cif_dim <= 512 && f->cif_hid <= 512 && f->affcif_hid <= 512 &&
                                        f->cif_hid > 0 && f->affcif_hid > 0 && !f->extra && !f->is_global));
    if (!dims_ok) { delete f; return FC_ERR_UNSUPPORTED; }
    f->layers = new (std::nothrow) FcFlowLayer[f->L];
    if (!f->layers) { delete f; return FC_ERR_MODEL; }

    FcCursor c{table, n_table, 0, arena, arena_floats, true};
    c.tc_fmt = header[1] == FC_ARENA_VERSION_F16 ? 1 : 0;
    const int64_t cbits = c.next();
    memcpy(&f->ldj_const, &cbits, sizeof(double));
    const int attn_k2 = f->is_global ? 0 : f->inner;
    if (f->has_aug) {
        if (!f->is_global) {
            f->augpre = c.mlp(f->d_in, 0, f->augpre_hid, f->n_augpre_hid, f->attn_in);
            f->augpre.act = f->act;
            f->augattn = read_attn(c, *f);
        }
        f->aug = c.mlp(f->d_in, attn_k2, f->aug_hid, f->n_aug_hid, 2 * (f->D - f->d_in));
        f->aug.act = f->act;
    }
    const int cpl_out = f->cpl_kind == FC_CPL_AFFINE ? 2 * n2 : f->cpl_kind == FC_CPL_SPLINE ? (3 * f->num_bins + 1) * f->half
                                                                                              : n2 * n2 + n2;
    f->has_cb = f->extra || f->is_global;
    if (f->has_cb) f->cb = c.linear(f->extra + (f->is_global ? f->E : 0), 0, (f->L + 1) * f->hid);
    for (int l = 0; l < f->L; ++l) {
        FcFlowLayer& y = f->layers[l];
        if (f->cif_dim) {
            y.cifnet = c.mlp(f->D, 0, f->cif_hid, f->n_cif_hid, 2 * S);                 // GELU (cif_block.py:54)
            y.affcif = c.mlp(S, 0, f->affcif_hid, f->n_affcif_hid, 2 * f->D);           // GELU (cif_block.py:64)
            y.cif_sc = c.ptr(c.next(), f->cif_dim);
            y.cif_bi = c.ptr(c.next(), f->cif_dim);
            if (!y.cif_sc || !y.cif_bi) c.ok = false;
        }
        if (!f->is_global) {
            y.pre = c.mlp(f->half, 0, f->pre_hid, f->n_pre_hid, f->attn_in);
            y.pre.act = f->cif_dim ? FC_ACT_GELU : f->act;                              // the CIF block's own MLP is GELU (:62)
            y.attn = read_attn(c, *f);
        }
        if (f->cpl_kind == FC_CPL_EXPO) { y.expo_sq = c.ptr(c.next(), 4); if (!y.expo_sq) c.ok = false; }
        y.cpl = c.mlp(f->half, attn_k2, f->hid, f->n_hid, cpl_out);
        y.cpl.act = f->act;
        y.has_lu = (l != f->L - 1);
        if (y.has_lu) {
            y.lu = c.linear(f->D, 0, f->D);
            y.lu_diag = c.ptr(c.next(), f->D);
            if (!y.lu_diag) c.ok = false;
        }
    }
    if (!c.ok || c.pos != n_table) { fc_flow_destroy(f); return FC_ERR_MODEL; }
    *out = f;
    return FC_OK;
}

extern "C" void fc_flow_destroy(fc_flow* f) {
    if (!f) return;
    delete[] f->layers;
    delete[] f->glayers;
    delete f;
}

// ------------------------------------------------------------------------------------------ workspace
namespace {
struct FlowWs {
    float *lat0, *lat1, *hA, *hB, *q, *o, *mu, *rstd, *cpart, *apart, *kv, *kvs, *cb, *cbA, *pbuf;
    int ldx, ldh, n_cpart, n_apart, cb_ld, cbA_ld, ldp, p_rows, ldp_cif;
    int64_t total_bytes;
};

FlowWs carve_flow_ws(const fc_flow* f, int B, int N, int Nc, void* base) {
    FlowWs w{};
    const int64_t M = (int64_t)B * N;
    w.ldx = fc_round_up(f->cif_dim > f->D ? f->cif_dim : f->D, 4);
    w.ldh = 512;
    // one partial log-det slab per N-tile of whichever GEMM kernel runs (FFMA: 128-wide tiles, tcgen05: <= 96-wide)
    auto slabs = [](int n) { const int a = fc_gemm_n_tiles(n), b = fc_tc_n_tiles(n); return a > b ? a : b; };
    w.n_cpart = slabs(2 * (f->D - f->half));
    if (f->cif_dim) { const int a = slabs(2 * f->D); if (a > w.n_cpart) w.n_cpart = a; }
    w.n_apart = f->has_aug ? slabs(2 * (f->D - f->d_in)) : 1;
    // raw conditioner outputs of the spline / exponential couplings and of the CIF block's ConditionalNormal net; the
    // exponential coupling's (n^2 + n floats per point) are produced and consumed in chunks of whole clouds
    w.ldp = 0; w.p_rows = 0; w.ldp_cif = 0;
    {
        const int n2 = f->D - f->half;
        if (f->cpl_kind == FC_CPL_SPLINE) { w.ldp = fc_round_up((3 * f->num_bins + 1) * f->half, 4); w.p_rows = (int)M; }
        if (f->cpl_kind == FC_CPL_EXPO) {
            w.ldp = fc_round_up(n2 * n2 + n2, 4);
            const long long clouds = (1ll << 28) / ((long long)w.ldp * N);     // ~1 GB of parameters at a time
            w.p_rows = (int)((clouds < 1 ? 1 : (clouds > B ? B : clouds)) * N);
        }
        if (f->cif_dim) w.ldp_cif = fc_round_up(2 * (f->cif_dim - f->D), 4);
    }
    w.cb_ld = (f->L + 1) * f->hid;
    w.cbA_ld = fc_round_up(f->extra + (f->is_global ? f->E : 0), 4);
    if (w.cbA_ld == 0) w.cbA_ld = 4;
    int64_t off = 0;
    auto take = [&](int64_t floats) { float* p = base ? reinterpret_cast<float*>(reinterpret_cast<char*>(base) + off) : nullptr;
                                      off += fc_round_up_ll(floats * 4, 256); return p; };
    w.lat0 = take(M * w.ldx); w.lat1 = take(M * w.ldx);
    w.hA = take(M * w.ldh); w.hB = take(M * w.ldh);
    w.q = take(M * 64); w.o = take(M * 64);
    w.mu = take(M); w.rstd = take(M);
    w.cpart = take(M * w.n_cpart); w.apart = take(M * w.n_apart);
    // attention configs only (the global embedder's flow never runs an attention kernel)
    w.kv = take(f->is_global ? 0 : (int64_t)B * Nc * 128);
    w.kvs = take(f->is_global ? 0 : fc_attention_tc_scratch_floats(B, Nc));   // TF32 hi/lo copies of k, v^T for the tcgen05 attention
    w.cb = take((int64_t)B * w.cb_ld);
    w.cbA = take((int64_t)B * w.cbA_ld);
    {
        const int64_t a = (int64_t)w.ldp * w.p_rows, b = (int64_t)w.ldp_cif * M;
        w.pbuf = take(a > b ? a : b);
    }
    w.total_bytes = off;
    return w;
}
}  // namespace

extern "C" int64_t fc_flow_workspace_bytes(const fc_flow* f, int B, int N, int Nc) {
    if (!f || B <= 0 || N <= 0 || Nc <= 0) return FC_ERR_INVALID_ARG;
    return carve_flow_ws(f, B, N, Nc, nullptr).total_bytes;
}

// ------------------------------------------------------------------------------------------ forward
// Which attention blocks' softmax weights a forward pass writes (fc_flow_attention_maps), or whose score gradients the
// input-gradient pass writes (fc_flow_attention_score_grads).  Slot 0 is the augmenter's attention, slot l + 1 coupling layer
// l's; `slots` strictly increasing; the i-th captured block's maps [B, n_query, Nc] start at out + i * B * n_query * Nc, or,
// with `accumulate` (score gradients only), every block adds into the one [B, n_query, Nc] at out.
struct FcCapture { const int32_t* slots; int n_slots; const int32_t* qidx; int n_query; float* out; bool accumulate; };

// a caller's workspace: 256-byte aligned and at least `need` bytes
static bool ws_ok(const void* workspace, int64_t need, int64_t workspace_bytes) {
    return workspace && !(reinterpret_cast<uintptr_t>(workspace) & 255) && need <= workspace_bytes;
}

// LayerNorm statistics, to_q, to_kv and the attention of one block, from its pre-attention MLP's output h4 [M][ldh4]: w.o
// (and w.q, w.mu, w.rstd) afterwards.  maps: where this block's weights go (nullptr: not captured; `cap` then unused)
static int run_attention_core(const fc_flow* f, const FcAttn& at, const float* h4, int ldh4, const float* context, int B, int N,
                              int Nc, FlowWs& w, int precision, cudaStream_t s, float* maps, const FcCapture* cap) {
    const int M = B * N;
    int rc = fc_launch_ln_stats(h4, ldh4, M, f->attn_in, 1e-5f, w.mu, w.rstd, s);
    if (rc) return rc;
    {
        GemmArgs g = fc_gemm_linear(at.q, h4, ldh4, w.q, 64, M, precision);
        g.bias = at.qbias; g.epi = FC_EPI_LNQ; g.row_mu = w.mu; g.row_rstd = w.rstd; g.csum = at.csum;
        rc = fc_launch_gemm(g, s);
        if (rc) return rc;
    }
    // reference models/perceiver.py:104: scale = inner_dim ** -0.5
    const float scale = 1.0f / sqrtf((float)f->inner);
    const GemmArgs kv = fc_gemm_linear(at.kv, context, f->E, w.kv, 128, B * Nc, precision);
    if (maps) {
        // k through the plain epilogue into w.kv: the forward's own to_kv below either rewrites w.kv with the same values or
        // (tensor-core path) writes its split copies elsewhere and never reads it, so the forward is unchanged by the capture
        rc = fc_launch_gemm(kv, s);
        if (rc) return rc;
        rc = fc_launch_attention_maps(w.q, 64, w.kv, 128, cap->qidx, cap->n_query, maps, B, N, Nc, scale, s);
        if (rc) return rc;
    }
    if (precision == 1 && at.kv.N == 128 && at.kv.whi) {
        // to_kv writes the TF32 hi/lo copies of k and v^T the tcgen05 attention consumes, straight from its epilogue
        GemmArgs g = kv;
        g.epi = FC_EPI_KVSPLIT; g.ldc = 64; g.kv_nc = Nc;
        g.kv_f16 = at.kv.tc_fmt ? 1 : 0;      // 3xFP16 models run the attention on fp16 operands as well
        fc_attention_tc_scratch_layout(B, Nc, w.kvs, &g.C, &g.kv_klo, &g.kv_vthi, &g.kv_vtlo, &g.kv_ncp, g.kv_f16);
        rc = fc_launch_gemm(g, s);
        if (rc) return rc;
        return fc_launch_cross_attention_tc(w.q, 64, nullptr, 0, w.o, 64, B, N, Nc, f->inner, scale, w.kvs, 1, g.kv_f16, s);
    }
    rc = fc_launch_gemm(kv, s);
    if (rc) return rc;
    if (precision == 1)
        return fc_launch_cross_attention_tc(w.q, 64, w.kv, 128, w.o, 64, B, N, Nc, f->inner, scale, w.kvs, 0, at.kv.tc_fmt ? 1 : 0, s);
    return fc_launch_cross_attention(w.q, 64, w.kv, 128, w.o, 64, B, N, Nc, f->inner, scale, s);
}

// the pre-attention MLP on lat[:, :pre.in.K1], then run_attention_core
static int run_attention_block(const fc_flow* f, const FcMlp& pre, const FcAttn& at, const float* lat, int ldx,
                               const float* context, int B, int N, int Nc, FlowWs& w, int precision, cudaStream_t s,
                               float* maps = nullptr, const FcCapture* cap = nullptr) {
    const int M = B * N;
    FcMlpIn in{lat, ldx, nullptr, 0, nullptr, 0, 0};
    float* last = nullptr;
    int rc = fc_run_mlp_hidden(pre, in, M, w.hA, w.hB, w.ldh, precision, s, &last);
    if (rc) return rc;
    float* h4 = (last == w.hA) ? w.hB : w.hA;
    rc = fc_launch_gemm(fc_gemm_linear(pre.out, last, w.ldh, h4, w.ldh, M, precision), s);
    if (rc) return rc;
    return run_attention_core(f, at, h4, w.ldh, context, B, N, Nc, w, precision, s, maps, cap);
}

// per-cloud bias of every conditioner's first layer (extra context and/or global embedding) into w.cb
static int run_cb_prologue(const fc_flow* f, const float* extra, const float* context, int B, FlowWs& w, cudaStream_t s) {
    if (!f->has_cb) return FC_OK;
    const int tot = B * w.cbA_ld;
    build_cb_input_kernel<<<(tot + 255) / 256, 256, 0, s>>>(extra, context, f->E, f->extra, f->is_global, B, w.cbA_ld, w.cbA);
    fc_count_launch();
    FC_LAUNCH_OK();
    return fc_launch_gemm(fc_gemm_linear(f->cb, w.cbA, w.cbA_ld, w.cb, w.cb_ld, B, 0 /* always exact fp32: tiny */), s);
}

// the first layer's input of a conditioner (slot 0: the augmenter's, l + 1: coupling layer l's) over N points per cloud: the
// latent, the attention output (attention configs) and the per-cloud bias row of that slot
static FcMlpIn conditioner_in(const fc_flow* f, const FlowWs& w, const float* lat, int slot, int N) {
    FcMlpIn in{lat, w.ldx, f->is_global ? nullptr : w.o, 64, nullptr, 0, 0};
    if (f->has_cb) { in.bias = w.cb + (size_t)slot * f->hid; in.bias_ld = w.cb_ld; in.bias_group = N; }
    return in;
}

// an affine coupling in the epilogue of its conditioner's output GEMM, on latent columns from col0: x2 = x2 * s + t with the
// log-det partials in w.cpart, or (inverse) x2 = (x2 - t) / s
static int affine_coupling_gemm(const FcLinear& out, const float* last, float* lat, int col0, FlowWs& w, int M, int precision,
                                bool inverse, cudaStream_t s) {
    GemmArgs g = fc_gemm_linear(out, last, w.ldh, nullptr, 0, M, precision);
    g.epi = inverse ? FC_EPI_COUPLING_INV : FC_EPI_COUPLING;
    g.x = lat; g.ldx = w.ldx; g.col0 = col0; g.part = inverse ? nullptr : w.cpart;
    return fc_launch_gemm(g, s);
}

// ActNorm + LinearLU as one GEMM, dst = diag.src + (W' - diag) src + b': the diagonal (~1) is applied to the fp32 latent in the
// epilogue, the GEMM only carries the off-diagonal mixing, so its rounding (and the tensor core's accumulate truncation) acts on
// the small part instead of shrinking z itself 114 times in a row.  The same split serves the inverse and, on the transposed
// off-diagonal part, the input-gradient pass.
static int lu_gemm(const FcLinear& l, const float* diag, const float* src, float* dst, int ldx, int M, int precision,
                   cudaStream_t s) {
    GemmArgs g = fc_gemm_linear(l, src, ldx, dst, ldx, M, precision);
    g.res = src; g.ldres = ldx; g.res_scale = diag;
    return fc_launch_gemm(g, s);
}

// Coupling layer l on lat (N points per cloud), forward or inverse: the conditioner reads the untouched half x1 (and the
// attention output, the per-cloud bias) the same way in both directions; the transform then updates x2 = columns [half, D) in
// place, the forward writing its log-det partials to w.cpart.  maps / cap: attention capture as in run_attention_core.
static int run_coupling(const fc_flow* f, int l, float* lat, const float* context, int B, int N, int Nc, FlowWs& w, int precision,
                        bool inverse, cudaStream_t s, float* maps = nullptr, const FcCapture* cap = nullptr) {
    const FcFlowLayer& y = f->layers[l];
    const int M = B * N, n2 = f->D - f->half, inv = inverse ? 1 : 0;
    float* part = inverse ? nullptr : w.cpart;
    int rc;
    if (!f->is_global) {
        rc = run_attention_block(f, y.pre, y.attn, lat, w.ldx, context, B, N, Nc, w, precision, s, maps, cap);
        if (rc) return rc;
    }
    float* last = nullptr;
    rc = fc_run_mlp_hidden(y.cpl, conditioner_in(f, w, lat, l + 1, N), M, w.hA, w.hB, w.ldh, precision, s, &last);
    if (rc) return rc;
    if (f->cpl_kind == FC_CPL_SPLINE) {
        // reference models/spline_coupling.py:187-227: the conditioner's raw output, then the spline on x2 in place
        rc = fc_launch_gemm(fc_gemm_linear(y.cpl.out, last, w.ldh, w.pbuf, w.ldp, M, precision), s);
        if (rc) return rc;
        return fc_launch_rq_spline(w.pbuf, w.ldp, lat, w.ldx, f->half, n2, f->num_bins, M, part, inv, s);
    }
    if (f->cpl_kind == FC_CPL_EXPO) {
        // reference models/exponential_coupling.py:44-77, n^2 + n conditioner outputs per point: whole clouds at a time
        for (int r0 = 0; r0 < M; r0 += w.p_rows) {
            const int rows = M - r0 < w.p_rows ? M - r0 : w.p_rows;
            rc = fc_launch_gemm(fc_gemm_linear(y.cpl.out, last + (size_t)r0 * w.ldh, w.ldh, w.pbuf, w.ldp, rows, precision), s);
            if (rc) return rc;
            rc = fc_launch_expm_action(w.pbuf, w.ldp, lat, w.ldx, f->half, n2, y.expo_sq, part, r0, rows, inv, s);
            if (rc) return rc;
        }
        return FC_OK;
    }
    // reference models/affine_coupling.py:34-62
    return affine_coupling_gemm(y.cpl.out, last, lat, f->half, w, M, precision, inverse, s);
}

// CIF block up to (not including) its attention-conditioned coupling, reference models/cif_block.py:71-93.  In the
// reference's order: Augment -> Reverse -> AffineCoupling(split = cif_dim - D) -> ActNorm -> Reverse -> Slice.  The two
// Reverse permutations cancel once the affine coupling's weights and the ActNorm vectors are re-indexed at pack time
// (packing.py: _pack_cif), so on the device the block is: z2 ~ N(mean(x), sigma(x)) into columns [D, cif_dim);
// x = x * s(z2) + t(z2); every column c: a*sc[c] + bi[c]; log N(z2; mean(x), sigma(x)) with the SAME net (cif_block.py:58).
static int run_cif_block(const fc_flow* f, const FcFlowLayer& y, float* lat, FlowWs& w, int M, const float* eps_l,
                         int precision, cudaStream_t s) {
    const int D = f->D, S = f->cif_dim - f->D;
    int rc;
    for (int pass = 0; pass < 2; ++pass) {
        FcMlpIn in{lat, w.ldx, nullptr, 0, nullptr, 0, 0};
        float* last = nullptr;
        rc = fc_run_mlp_hidden(y.cifnet, in, M, w.hA, w.hB, w.ldh, precision, s, &last);
        if (rc) return rc;
        rc = fc_launch_gemm(fc_gemm_linear(y.cifnet.out, last, w.ldh, w.pbuf, w.ldp_cif, M, precision), s);
        if (rc) return rc;
        rc = fc_launch_cond_normal(w.pbuf, w.ldp_cif, lat, w.ldx, D, S, eps_l, M, f->cif_clamp, w.cpart, pass, s);
        if (rc || pass == 1) return rc;
        FcMlpIn in2{lat + D, w.ldx, nullptr, 0, nullptr, 0, 0};
        rc = fc_run_mlp_hidden(y.affcif, in2, M, w.hA, w.hB, w.ldh, precision, s, &last);
        if (rc) return rc;
        rc = affine_coupling_gemm(y.affcif.out, last, lat, 0, w, M, precision, false, s);
        if (rc) return rc;
        rc = fc_launch_col_affine(lat, w.ldx, f->cif_dim, M, y.cif_sc, y.cif_bi, s);
        if (rc) return rc;
    }
    return FC_OK;
}

// draws > 0: the K-draw pass of fc_flow_log_prob_draws.  The augmenter's network depends on (x, c) only, so it runs once over
// the B*N points with x staged in lat1; its output GEMM then runs once per draw (eps + k*B*N*S) into that staging latent and
// staging log-det slabs, and fc_launch_scatter_draw moves the result to rows (b*K + k)*N + n of lat0 / apart.  Every later
// layer runs unchanged on K*N points per cloud.  Each launch a row goes through is the launch log_prob makes for it, so draw k
// is bitwise fc_flow_log_prob with eps + k*B*N*S.  eps_cif is then [L, B, K, N, S]; log_prob_out [K, B, N].
static int flow_forward(const fc_flow* f, const float* x, const float* context, const float* extra, const float* eps,
                        const float* eps_cif, float* log_prob_out, float* z_out, int B, int N, int Nc, void* workspace,
                        int64_t workspace_bytes, int precision, fc_stream_t stream_, const FcCapture* cap = nullptr,
                        int draws = 0, float* ckpt = nullptr) {
    FC_REQUIRE(f && x && context && log_prob_out && B > 0 && N > 0 && Nc > 0 && draws >= 0);
    FC_REQUIRE(!ckpt || !draws);
    FC_REQUIRE(eps || !f->has_aug);
    FC_REQUIRE(eps_cif || !f->cif_dim);
    FC_REQUIRE((f->extra != 0) == (extra != nullptr));
    FC_REQUIRE(!draws || (!cap && !z_out));
    const int K = draws ? draws : 1;
    FC_REQUIRE((int64_t)B * N * K < (1ll << 31) && (int64_t)B * Nc < (1ll << 31));
    cudaStream_t s = (cudaStream_t)stream_;
    FlowWs w = carve_flow_ws(f, B, K * N, Nc, workspace);
    if (!ws_ok(workspace, w.total_bytes, workspace_bytes)) return FC_ERR_WORKSPACE;
    const int NK = K * N;            // points per cloud after the augmenter
    const int M = B * NK, M0 = B * N;
    float* xin = draws ? w.lat1 : w.lat0;     // the latent the augmenter reads x from and writes its draw into
    int rc;

    // x -> latent columns [0, d_in)
    if ((rc = copy_cols(x, f->d_in, xin, w.ldx, M0, f->d_in, s))) return rc;
    // partial log-det slabs: the FFMA and tcgen05 GEMMs tile N differently (128 vs <=256 wide), so slabs a
    // path does not write must read as zero in finalize
    FC_CUDA_OK(cudaMemsetAsync(w.cpart, 0, (size_t)M * w.n_cpart * sizeof(float), s));
    FC_CUDA_OK(cudaMemsetAsync(w.apart, 0, (size_t)M * w.n_apart * sizeof(float), s));
    if ((rc = run_cb_prologue(f, extra, context, B, w, s))) return rc;
    int n_captured = 0;
    auto maps_for = [&](int slot) -> float* {
        if (!cap || n_captured >= cap->n_slots || cap->slots[n_captured] != slot) return nullptr;
        return cap->out + (size_t)(n_captured++) * (size_t)B * (size_t)cap->n_query * (size_t)Nc;
    };

    // ---- transforms.0: augment (reference models/augmenter.py:15-19, :49-63); latent_dim == input_dim: IdentityTransform
    if (f->has_aug && !f->is_global) {
        rc = run_attention_block(f, f->augpre, f->augattn, xin, w.ldx, context, B, N, Nc, w, precision, s, maps_for(0), cap);
        if (rc) return rc;
    }
    if (f->has_aug) {
        float* last = nullptr;
        rc = fc_run_mlp_hidden(f->aug, conditioner_in(f, w, xin, 0, N), M0, w.hA, w.hB, w.ldh, precision, s, &last);
        if (rc) return rc;
        GemmArgs g = fc_gemm_linear(f->aug.out, last, w.ldh, nullptr, 0, M0, precision);
        g.epi = FC_EPI_AUGMENT; g.x = xin; g.ldx = w.ldx; g.col0 = f->d_in;
        g.part = w.apart; g.eps = eps; g.ld_eps = f->D - f->d_in;
        if (!draws) {
            rc = fc_launch_gemm(g, s);
            if (rc) return rc;
        } else {
            // staging slabs in the hidden buffer the output GEMM does not read; slabs the GEMM path leaves alone stay zero
            float* spart = last == w.hA ? w.hB : w.hA;
            FC_CUDA_OK(cudaMemsetAsync(spart, 0, (size_t)M0 * w.n_apart * sizeof(float), s));
            g.part = spart;
            for (int k = 0; k < K; ++k) {
                g.eps = eps + (size_t)k * M0 * (f->D - f->d_in);
                rc = fc_launch_gemm(g, s);
                if (rc) return rc;
                rc = fc_launch_scatter_draw(xin, w.ldx, f->D, spart, w.n_apart, w.lat0, w.ldx, w.apart, B, N, K, k, s);
                if (rc) return rc;
            }
        }
    } else if (draws) {
        for (int k = 0; k < K; ++k) {    // identity augmenter (a CIF flow): the K copies of x
            rc = fc_launch_scatter_draw(xin, w.ldx, f->D, nullptr, 0, w.lat0, w.ldx, nullptr, B, N, K, k, s);
            if (rc) return rc;
        }
    }

    // ---- coupling layers
    float* lat = w.lat0; float* lat_next = w.lat1;
    // ckpt (input-gradient pass): the latent at the input of layer l into slot l of [L+1][M][ldx], the final latent into slot L --
    // copied before the coupling updates x2 in place; the forward's own launches are unchanged
    auto checkpoint = [&](int slot) -> int {
        if (ckpt)
            FC_CUDA_OK(cudaMemcpyAsync(ckpt + (size_t)slot * M * w.ldx, lat, (size_t)M * w.ldx * sizeof(float),
                                       cudaMemcpyDeviceToDevice, s));
        return FC_OK;
    };
    for (int l = 0; l < f->L; ++l) {
        const FcFlowLayer& y = f->layers[l];
        if ((rc = checkpoint(l))) return rc;
        if (f->cif_dim) {
            rc = run_cif_block(f, y, lat, w, M, eps_cif + (size_t)l * M * (f->cif_dim - f->D), precision, s);
            if (rc) return rc;
        }
        rc = run_coupling(f, l, lat, context, B, NK, Nc, w, precision, false, s, maps_for(l + 1), cap);
        if (rc) return rc;
        if (y.has_lu) {
            rc = lu_gemm(y.lu, y.lu_diag, lat, lat_next, w.ldx, M, precision, s);
            if (rc) return rc;
            float* t = lat; lat = lat_next; lat_next = t;
        }
    }
    if ((rc = checkpoint(f->L))) return rc;
    {
        const int wpb = 8;
        finalize_kernel<<<(M + wpb - 1) / wpb, wpb * 32, 0, s>>>(lat, w.ldx, f->D, w.apart, w.n_apart, w.cpart, w.n_cpart,
                                                                 M, (float)f->ldj_const, log_prob_out, N, K);
        fc_count_launch();
        FC_LAUNCH_OK();
    }
    if (z_out) return copy_cols(lat, w.ldx, z_out, f->D, M, f->D, s);   // the final latent, [B*N, D] contiguous
    return FC_OK;
}

extern "C" int fc_flow_log_prob(const fc_flow* f, const float* x, const float* context, const float* extra,
                                const float* eps, float* log_prob_out, int B, int N, int Nc, void* workspace,
                                int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    return flow_forward(f, x, context, extra, eps, nullptr, log_prob_out, nullptr, B, N, Nc, workspace, workspace_bytes, precision, stream_);
}

// Same pass for flows built with CIF blocks (latent_dim < cif_latent_dim): `eps_cif` [L, B, N, cif_latent_dim - latent_dim] holds
// the draw of every block's augmenter (reference models/cif_block.py:74), in transform-list order.
extern "C" int fc_flow_log_prob_cif(const fc_flow* f, const float* x, const float* context, const float* extra,
                                    const float* eps, const float* eps_cif, float* log_prob_out, int B, int N, int Nc,
                                    void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    return flow_forward(f, x, context, extra, eps, eps_cif, log_prob_out, nullptr, B, N, Nc, workspace, workspace_bytes, precision, stream_);
}

// No stochastic transform (identity augmenter, no CIF block): every draw is the same log_prob, computed once.
static bool flow_is_deterministic(const fc_flow* f) { return !f->has_aug && !f->cif_dim; }

extern "C" int64_t fc_flow_log_prob_draws_workspace_bytes(const fc_flow* f, int B, int N, int Nc, int K) {
    if (!f || B <= 0 || N <= 0 || Nc <= 0 || K <= 0) return FC_ERR_INVALID_ARG;
    if (flow_is_deterministic(f)) K = 1;
    if ((int64_t)K * B * N > FC_DRAWS_MAX_ROWS) return FC_ERR_INVALID_ARG;
    return carve_flow_ws(f, B, K * N, Nc, nullptr).total_bytes;
}

// K augmentation draws of every point in one pass (flow_forward with draws = K): lp_draws_out[k] is bitwise what
// fc_flow_log_prob(_cif) returns with eps + k*B*N*S (and draw k's CIF noise).
extern "C" int fc_flow_log_prob_draws(const fc_flow* f, const float* x, const float* context, const float* extra,
                                      const float* eps, const float* eps_cif, int K, float* lp_draws_out, int B, int N, int Nc,
                                      void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    FC_REQUIRE(f && K > 0 && B > 0 && N > 0 && lp_draws_out);
    if (flow_is_deterministic(f)) {
        FC_REQUIRE((int64_t)B * N <= FC_DRAWS_MAX_ROWS);
        const int rc = flow_forward(f, x, context, extra, eps, nullptr, lp_draws_out, nullptr, B, N, Nc, workspace,
                                    workspace_bytes, precision, stream_);
        if (rc) return rc;
        const size_t bytes = (size_t)B * N * sizeof(float);
        for (int k = 1; k < K; ++k)
            FC_CUDA_OK(cudaMemcpyAsync(lp_draws_out + (size_t)k * B * N, lp_draws_out, bytes, cudaMemcpyDeviceToDevice,
                                       (cudaStream_t)stream_));
        return FC_OK;
    }
    FC_REQUIRE((int64_t)K * B * N <= FC_DRAWS_MAX_ROWS);
    return flow_forward(f, x, context, extra, eps, eps_cif, lp_draws_out, nullptr, B, N, Nc, workspace, workspace_bytes, precision,
                        stream_, nullptr, K);
}

// The forward pass that also writes the softmax weights of the attention blocks listed in slots_host (see FcCapture).
extern "C" int fc_flow_attention_maps(const fc_flow* f, const float* x, const float* context, const float* extra, const float* eps,
                                      const float* eps_cif, const int32_t* slots_host, int n_slots, const int32_t* query_idx,
                                      int n_query, float* maps_out, float* log_prob_out, int B, int N, int Nc, void* workspace,
                                      int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    FC_REQUIRE(f && slots_host && n_slots > 0 && maps_out && n_query > 0);
    if (f->is_global) return FC_ERR_UNSUPPORTED;       // no attention over context points: the device never runs one
    FC_REQUIRE(query_idx || n_query == N);
    for (int i = 0; i < n_slots; ++i)
        FC_REQUIRE(slots_host[i] >= 0 && slots_host[i] <= f->L && (i == 0 || slots_host[i] > slots_host[i - 1]));
    FC_REQUIRE(slots_host[0] != 0 || f->has_aug);     // an identity augmenter has no attention
    const FcCapture cap{slots_host, n_slots, query_idx, n_query, maps_out, false};
    return flow_forward(f, x, context, extra, eps, eps_cif, log_prob_out, nullptr, B, N, Nc, workspace, workspace_bytes, precision,
                        stream_, &cap);
}

extern "C" int fc_flow_cif_noise_dim(const fc_flow* f) { return f ? (f->cif_dim ? f->cif_dim - f->D : 0) : FC_ERR_INVALID_ARG; }

extern "C" int fc_flow_forward(const fc_flow* f, const float* x, const float* context, const float* extra, const float* eps,
                               float* log_prob_out, float* z_out, int B, int N, int Nc, void* workspace, int64_t workspace_bytes,
                               int precision, fc_stream_t stream_) {
    FC_REQUIRE(z_out != nullptr);
    return flow_forward(f, x, context, extra, eps, nullptr, log_prob_out, z_out, B, N, Nc, workspace, workspace_bytes, precision, stream_);
}

// ------------------------------------------------------------------------------------------ inverse / sampling pass
extern "C" int fc_flow_set_inverse(fc_flow* f, const int32_t* header, int n_header, const int64_t* table, int n_table,
                                   const float* arena, int64_t arena_floats) {
    FC_REQUIRE(f && header && table && arena && n_header >= 4);
    if (header[0] != FC_INV_MAGIC || (header[1] != FC_ARENA_VERSION && header[1] != FC_ARENA_VERSION_F16)) return FC_ERR_MODEL;
    if (header[2] != f->L || header[3] != f->D || (reinterpret_cast<uintptr_t>(arena) & 15)) return FC_ERR_MODEL;
    if ((n_header >= 5 ? header[4] : 0) != f->cif_dim) return FC_ERR_MODEL;
    FcCursor c{table, n_table, 0, arena, arena_floats, true};
    c.tc_fmt = header[1] == FC_ARENA_VERSION_F16 ? 1 : 0;
    for (int l = 0; l < f->L; ++l) {
        FcFlowLayer& y = f->layers[l];
        if (f->cif_dim) {
            y.cif_isc = c.ptr(c.next(), f->cif_dim);
            y.cif_ibi = c.ptr(c.next(), f->cif_dim);
            if (!y.cif_isc || !y.cif_ibi) c.ok = false;
        }
        if (!y.has_lu) continue;
        y.lu_inv = c.linear(f->D, 0, f->D);
        y.lu_inv_diag = c.ptr(c.next(), f->D);
        if (!y.lu_inv_diag) c.ok = false;
    }
    if (!c.ok || c.pos != n_table) return FC_ERR_MODEL;
    f->has_inverse = true;
    return FC_OK;
}

// `Flow.sample` after the base draw (reference models/transform.py:79-84): the transform list walked backwards with each
// `.inverse` -- LinearLU (models/permuters.py:171-177) and ActNorm (models/act_norm.py:45-46) as ONE folded GEMM
// z = Wp^-1 z' + shift (packing.fold_inverse_actnorm_lu), the affine coupling's inverse x2 = (y2 - t)/s
// (models/affine_coupling.py:48-62) in the epilogue of its conditioner's last GEMM, the conditioner itself exactly as in the
// forward pass (it reads the untouched half y1); the augmenter's inverse keeps the first input_dim columns
// (models/augmenter.py:20-21,65-67).  z: [B, P, D] base draw, x_out: [B, P, d_in].
static int flow_sample(const fc_flow* f, const float* z, const float* context, const float* extra, const float* eps_cif,
                       float* x_out, int B, int P, int Nc, void* workspace, int64_t workspace_bytes, int precision,
                       fc_stream_t stream_) {
    FC_REQUIRE(f && z && context && x_out && B > 0 && P > 0 && Nc > 0);
    FC_REQUIRE((f->extra != 0) == (extra != nullptr));
    FC_REQUIRE(eps_cif || !f->cif_dim);
    FC_REQUIRE((int64_t)B * P < (1ll << 31) && (int64_t)B * Nc < (1ll << 31));
    if (!f->has_inverse) return FC_ERR_MODEL;
    cudaStream_t s = (cudaStream_t)stream_;
    FlowWs w = carve_flow_ws(f, B, P, Nc, workspace);
    if (!ws_ok(workspace, w.total_bytes, workspace_bytes)) return FC_ERR_WORKSPACE;
    const int M = B * P, S = f->cif_dim ? f->cif_dim - f->D : 0;
    int rc;
    if ((rc = copy_cols(z, f->D, w.lat0, w.ldx, M, f->D, s))) return rc;
    if ((rc = run_cb_prologue(f, extra, context, B, w, s))) return rc;
    float* lat = w.lat0; float* lat_next = w.lat1;
    for (int l = f->L - 1; l >= 0; --l) {
        const FcFlowLayer& y = f->layers[l];
        if (y.has_lu) {
            rc = lu_gemm(y.lu_inv, y.lu_inv_diag, lat, lat_next, w.ldx, M, precision, s);
            if (rc) return rc;
            float* t = lat; lat = lat_next; lat_next = t;
        }
        rc = run_coupling(f, l, lat, context, B, P, Nc, w, precision, true, s);
        if (rc) return rc;
        if (f->cif_dim) {
            // CIFblock.inverse after its flow (reference models/cif_block.py:102-111), Reverse folded as in the forward pass:
            // the sliced-off columns are SAMPLED from the ConditionalNormal of what was kept (models/slice.py:46-58), then the
            // inverse ActNorm on all cif_dim columns and x = (x - t(z2)) / s(z2); Augment.inverse drops the extra columns.
            FcMlpIn inc{lat, w.ldx, nullptr, 0, nullptr, 0, 0};
            float* last = nullptr;
            rc = fc_run_mlp_hidden(y.cifnet, inc, M, w.hA, w.hB, w.ldh, precision, s, &last);
            if (rc) return rc;
            rc = fc_launch_gemm(fc_gemm_linear(y.cifnet.out, last, w.ldh, w.pbuf, w.ldp_cif, M, precision), s);
            if (rc) return rc;
            rc = fc_launch_cond_normal(w.pbuf, w.ldp_cif, lat, w.ldx, f->D, S, eps_cif + (size_t)l * M * S, M, f->cif_clamp,
                                       w.cpart /* log-density not needed: scratch */, 0, s);
            if (rc) return rc;
            rc = fc_launch_col_affine(lat, w.ldx, f->cif_dim, M, y.cif_isc, y.cif_ibi, s);
            if (rc) return rc;
            FcMlpIn in2{lat + f->D, w.ldx, nullptr, 0, nullptr, 0, 0};
            rc = fc_run_mlp_hidden(y.affcif, in2, M, w.hA, w.hB, w.ldh, precision, s, &last);
            if (rc) return rc;
            rc = affine_coupling_gemm(y.affcif.out, last, lat, 0, w, M, precision, true, s);
            if (rc) return rc;
        }
    }
    return copy_cols(lat, w.ldx, x_out, f->d_in, M, f->d_in, s);
}

extern "C" int fc_flow_sample(const fc_flow* f, const float* z, const float* context, const float* extra, float* x_out, int B,
                              int P, int Nc, void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    return flow_sample(f, z, context, extra, nullptr, x_out, B, P, Nc, workspace, workspace_bytes, precision, stream_);
}

// Flows with CIF blocks: eps_cif [L, B, P, fc_flow_cif_noise_dim(f)] = the N(0,1) draws of every block's `Slice.inverse`
// (reference models/slice.py:46-58), indexed by the block's position in the FORWARD list.
extern "C" int fc_flow_sample_cif(const fc_flow* f, const float* z, const float* context, const float* extra,
                                  const float* eps_cif, float* x_out, int B, int P, int Nc, void* workspace,
                                  int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    return flow_sample(f, z, context, extra, eps_cif, x_out, B, P, Nc, workspace, workspace_bytes, precision, stream_);
}

// ------------------------------------------------------------------------------------------ input-gradient pass
// d log_prob / d x of `Flow.log_prob` (reference models/transform.py:70-76) with eps held fixed, for affine-coupling flows.
// The forward pass runs unchanged and copies the latent at the input of every coupling layer into a checkpoint slab; the layers
// are then walked backwards: each one's forward is recomputed from its checkpoint with the intermediates its backward needs
// (pre-activations, the LayerNorm input and statistics, q, the attention output, the raw coupling outputs), then its backward
// runs.  Every backward contraction is a GEMM on the transposed weights fc_flow_set_grad attaches; the rest is flow_grad.cu.
static FcMlpT read_mlp_t(FcCursor& c, int K_x, bool has_o, int hid, int n_hidden, int N_out) {
    FcMlpT t;
    if (n_hidden > FC_MAX_HIDDEN) { c.ok = false; return t; }
    t.in_x = c.linear(hid, 0, K_x, false);
    if (has_o) t.in_o = c.linear(hid, 0, 64, false);
    for (int i = 0; i < n_hidden; ++i) t.hidden[i] = c.linear(hid, 0, hid, false);
    t.out = c.linear(N_out, 0, hid, false);
    return t;
}

extern "C" int fc_flow_set_grad(fc_flow* f, const int32_t* header, int n_header, const int64_t* table, int n_table,
                                const float* arena, int64_t arena_floats) {
    FC_REQUIRE(f && header && table && arena && n_header >= 4);
    if (f->cpl_kind != FC_CPL_AFFINE || f->cif_dim) return FC_ERR_UNSUPPORTED;
    if (header[0] != FC_GRAD_MAGIC || header[1] != FC_ARENA_VERSION) return FC_ERR_MODEL;
    if (header[2] != f->L || header[3] != f->D || (reinterpret_cast<uintptr_t>(arena) & 15)) return FC_ERR_MODEL;
    FcGradLayer* gl = new (std::nothrow) FcGradLayer[f->L];
    if (!gl) return FC_ERR_MODEL;
    FcGradLayer ga;
    FcCursor c{table, n_table, 0, arena, arena_floats, true};
    c.tc_fmt = 0;                                     // transposed weights: 3xTF32 copies whatever the model's format
    const bool attn = !f->is_global;
    if (f->has_aug) {
        if (attn) {
            ga.pre = read_mlp_t(c, f->d_in, false, f->augpre_hid, f->n_augpre_hid, f->attn_in);
            ga.q = c.linear(f->inner, 0, f->attn_in, false);
        }
        ga.cpl = read_mlp_t(c, f->d_in, attn, f->aug_hid, f->n_aug_hid, 2 * (f->D - f->d_in));
    }
    for (int l = 0; l < f->L; ++l) {
        FcGradLayer& y = gl[l];
        if (attn) {
            y.pre = read_mlp_t(c, f->half, false, f->pre_hid, f->n_pre_hid, f->attn_in);
            y.q = c.linear(f->inner, 0, f->attn_in, false);
        }
        y.cpl = read_mlp_t(c, f->half, attn, f->hid, f->n_hid, 2 * (f->D - f->half));
        if (f->layers[l].has_lu) y.lu = c.linear(f->D, 0, f->D, false);
    }
    if (!c.ok || c.pos != n_table) { delete[] gl; return FC_ERR_MODEL; }
    delete[] f->glayers;
    f->glayers = gl;
    f->gaug = ga;
    return FC_OK;
}

namespace {
struct GradWs {
    FlowWs fw;                                // the forward pass's own workspace (its buffers are reused by the recompute)
    float* ckpt;                              // [L+1][M][ldx]
    float *gA, *gB;                           // dL/d(latent), [M][ldx]
    float* ppre[FC_MAX_HIDDEN + 1];           // pre-activations of the pre-attention MLP's in / hidden layers, [M][ldh]
    float* cpre[FC_MAX_HIDDEN + 1];           // ... of the coupling (augmenter) MLP's
    float* post[3];                           // activations of the recompute (h_i in post[i % 3])
    float *h4, *dA, *dB, *raw, *dst, *dq, *dO;
    int ldr;
    int64_t total_bytes;
};

GradWs carve_grad_ws(const fc_flow* f, int B, int N, int Nc, void* base) {
    GradWs g{};
    g.fw = carve_flow_ws(f, B, N, Nc, base);
    const int64_t M = (int64_t)B * N;
    const int ldx = g.fw.ldx, ldh = g.fw.ldh;
    const int n2 = f->D - f->half;
    g.ldr = fc_round_up(2 * (n2 > f->D - f->d_in ? n2 : f->D - f->d_in), 4);
    int64_t off = g.fw.total_bytes;
    auto take = [&](int64_t floats) { float* p = base ? reinterpret_cast<float*>(reinterpret_cast<char*>(base) + off) : nullptr;
                                      off += fc_round_up_ll(floats * 4, 256); return p; };
    g.ckpt = take((int64_t)(f->L + 1) * M * ldx);
    g.gA = take(M * ldx); g.gB = take(M * ldx);
    const int np = f->is_global ? 0 : 1 + (f->n_pre_hid > f->n_augpre_hid ? f->n_pre_hid : f->n_augpre_hid);
    const int nc = 1 + (f->n_hid > f->n_aug_hid ? f->n_hid : f->n_aug_hid);
    for (int i = 0; i < np; ++i) g.ppre[i] = take(M * ldh);
    for (int i = 0; i < nc; ++i) g.cpre[i] = take(M * ldh);
    for (int i = 0; i < 3; ++i) g.post[i] = take(M * ldh);
    g.h4 = take(f->is_global ? 0 : M * ldh);
    g.dA = take(M * ldh); g.dB = take(M * ldh);
    g.raw = take(M * g.ldr); g.dst = take(M * g.ldr);
    g.dq = take(M * 64); g.dO = take(M * 64);
    g.total_bytes = off;
    return g;
}
}  // namespace

extern "C" int64_t fc_flow_log_prob_grad_workspace_bytes(const fc_flow* f, int B, int N, int Nc) {
    if (!f || B <= 0 || N <= 0 || Nc <= 0 || (int64_t)B * N > FC_GRAD_MAX_ROWS) return FC_ERR_INVALID_ARG;
    return carve_grad_ws(f, B, N, Nc, nullptr).total_bytes;
}

// whether fc_launch_gemm runs this GEMM on the tcgen05 path (whose epilogue evaluates GELU with fc_gelu_erf_fast)
static bool runs_on_tc(const GemmArgs& g) { return g.precision == 1 && fc_gemm_tc_supported(g); }

// fc_run_mlp_hidden with every layer's pre-activation kept: the GEMM stores act's argument (residual included) in pre[i], the
// forward's own activation for that GEMM path then gives h_i in post[i % 3].  Bitwise the forward's activations.
static int mlp_recompute(const FcMlp& m, const FcMlpIn& in, int M, float* const* pre, float* const* post, int ldh, int precision,
                         cudaStream_t s, const float** last) {
    GemmArgs g = mlp_in_gemm(m, in, pre[0], ldh, M, precision);
    int rc = fc_launch_gemm(g, s);
    if (rc) return rc;
    rc = fc_launch_act_fwd(pre[0], ldh, post[0], ldh, M, m.in.N, m.act, runs_on_tc(g), s);
    if (rc) return rc;
    for (int i = 0; i < m.n_hidden; ++i) {
        g = fc_gemm_linear(m.hidden[i], post[i % 3], ldh, pre[i + 1], ldh, M, precision);
        if (i & 1) { g.res = post[(i + 2) % 3]; g.ldres = ldh; }     // odd i: h_{i-1} (reference models/nets.py:19-30)
        rc = fc_launch_gemm(g, s);
        if (rc) return rc;
        rc = fc_launch_act_fwd(pre[i + 1], ldh, post[(i + 1) % 3], ldh, M, m.hidden[i].N, m.act, runs_on_tc(g), s);
        if (rc) return rc;
    }
    *last = post[m.n_hidden % 3];
    return FC_OK;
}

// Backward through an MLP's hidden layers.  On entry *cur holds dL/d h_n (the last activation), *other is free; on exit *cur
// holds dL/d pre_0.  Odd hidden layer i adds h_{i-1}: its dL/d pre_{i+1} stays in *other until it joins h_{i-1}'s gradient
// through the next GEMM's residual.
static int mlp_backward(const FcMlp& m, const FcMlpT& t, float* const* pre, int M, float** cur, float** other, int ldh,
                        int precision, cudaStream_t s) {
    const int hid = m.in.N;
    int rc;
    for (int i = m.n_hidden - 1; i >= 0; --i) {
        rc = fc_launch_act_bwd(*cur, ldh, pre[i + 1], ldh, M, hid, m.act, s);
        if (rc) return rc;
        GemmArgs g = fc_gemm_linear(t.hidden[i], *cur, ldh, *other, ldh, M, precision);
        if (!(i & 1) && i + 1 < m.n_hidden) { g.res = *other; g.ldres = ldh; }
        rc = fc_launch_gemm(g, s);
        if (rc) return rc;
        float* tmp = *cur; *cur = *other; *other = tmp;
    }
    return fc_launch_act_bwd(*cur, ldh, pre[0], ldh, M, hid, m.act, s);
}

// the forward of a pre-attention MLP and its attention block on lat[:, :pre.in.K1]: pre-activations in gw.ppre, the MLP's output
// in gw.h4, q / o / mu / rstd in gw.fw, and k / v through the plain epilogue in gw.fw.kv (the tensor-core attention reads split
// copies instead)
static int attn_recompute(const fc_flow* f, const FcMlp& pre, const FcAttn& at, const float* lat, int ldx, const float* context,
                          int B, int N, int Nc, GradWs& gw, int precision, cudaStream_t s) {
    const int M = B * N, ldh = gw.fw.ldh;
    FcMlpIn in{lat, ldx, nullptr, 0, nullptr, 0, 0};
    const float* last = nullptr;
    int rc = mlp_recompute(pre, in, M, gw.ppre, gw.post, ldh, precision, s, &last);
    if (rc) return rc;
    rc = fc_launch_gemm(fc_gemm_linear(pre.out, last, ldh, gw.h4, ldh, M, precision), s);
    if (rc) return rc;
    rc = run_attention_core(f, at, gw.h4, ldh, context, B, N, Nc, gw.fw, precision, s, nullptr, nullptr);
    if (rc) return rc;
    return fc_launch_gemm(fc_gemm_linear(at.kv, context, f->E, gw.fw.kv, 128, B * Nc, precision), s);
}

// with dL/do in gw.dO: dq, then LayerNorm and the pre-attention MLP backwards; g[:, :pre.in.K1] += dL/d(its input).
// sgrad: where this block's score gradients go (nullptr: not captured; `cap` then unused), added to it when sgrad_add.  They are
// read from q, k|v, o and dO as the dq kernel reads them, before anything else of the block's backward runs.
static int attn_backward(const fc_flow* f, const FcMlp& pre, const FcGradLayer& gl, int B, int N, int Nc, GradWs& gw, float* g,
                         int ldg, int precision, cudaStream_t s, float* sgrad, bool sgrad_add, const FcCapture* cap) {
    const int M = B * N, ldh = gw.fw.ldh;
    const float scale = 1.0f / sqrtf((float)f->inner);
    int rc;
    if (sgrad) {
        rc = fc_launch_attention_score_grad(gw.fw.q, 64, gw.fw.kv, 128, gw.fw.o, 64, gw.dO, 64, cap->qidx, cap->n_query, sgrad,
                                            sgrad_add ? 1 : 0, B, N, Nc, scale, s);
        if (rc) return rc;
    }
    rc = fc_launch_attention_dq(gw.fw.q, gw.fw.kv, 128, gw.fw.o, gw.dO, gw.dq, B, N, Nc, scale, s);
    if (rc) return rc;
    rc = fc_launch_gemm(fc_gemm_linear(gl.q, gw.dq, 64, gw.dA, ldh, M, precision), s);
    if (rc) return rc;
    rc = fc_launch_ln_bwd(gw.h4, ldh, gw.fw.mu, gw.fw.rstd, gw.dA, ldh, M, f->attn_in, s);
    if (rc) return rc;
    rc = fc_launch_gemm(fc_gemm_linear(gl.pre.out, gw.dA, ldh, gw.dB, ldh, M, precision), s);
    if (rc) return rc;
    float* cur = gw.dB; float* other = gw.dA;
    rc = mlp_backward(pre, gl.pre, gw.ppre, M, &cur, &other, ldh, precision, s);
    if (rc) return rc;
    GemmArgs a = fc_gemm_linear(gl.pre.in_x, cur, ldh, g, ldg, M, precision);
    a.res = g; a.ldres = ldg;
    return fc_launch_gemm(a, s);
}

// One conditioner (a coupling layer's, or the augmenter's with aug = true) backwards.  lat: the block's input (its checkpoint);
// g: dL/d(block output) on entry, dL/d(block input) on exit.  sgrad / sgrad_add / cap: score-gradient capture as in attn_backward.
static int conditioner_backward(const fc_flow* f, const FcMlp& pre, const FcAttn& at, const FcMlp& net, const FcGradLayer& gl,
                                bool aug, const float* lat, int cb_slot, const float* context, const float* eps, int B, int N, int Nc,
                                GradWs& gw, float* g, int precision, cudaStream_t s, float* sgrad, bool sgrad_add,
                                const FcCapture* cap) {
    const int M = B * N, ldh = gw.fw.ldh, ldx = gw.fw.ldx;
    const bool attn = !f->is_global;
    int rc;
    if (attn) {
        rc = attn_recompute(f, pre, at, lat, ldx, context, B, N, Nc, gw, precision, s);
        if (rc) return rc;
    }
    const float* last = nullptr;
    rc = mlp_recompute(net, conditioner_in(f, gw.fw, lat, cb_slot, N), M, gw.cpre, gw.post, ldh, precision, s, &last);
    if (rc) return rc;
    rc = fc_launch_gemm(fc_gemm_linear(net.out, last, ldh, gw.raw, gw.ldr, M, precision), s);
    if (rc) return rc;
    if (aug) rc = fc_launch_augment_tail_bwd(gw.raw, gw.ldr, eps, f->D - f->d_in, g, ldx, f->d_in, gw.dst, gw.ldr, M, s);
    else     rc = fc_launch_coupling_tail_bwd(gw.raw, gw.ldr, lat, ldx, g, ldx, f->half, f->D - f->half, gw.dst, gw.ldr, M, s);
    if (rc) return rc;
    rc = fc_launch_gemm(fc_gemm_linear(gl.cpl.out, gw.dst, gw.ldr, gw.dA, ldh, M, precision), s);
    if (rc) return rc;
    float* cur = gw.dA; float* other = gw.dB;
    rc = mlp_backward(net, gl.cpl, gw.cpre, M, &cur, &other, ldh, precision, s);
    if (rc) return rc;
    GemmArgs a = fc_gemm_linear(gl.cpl.in_x, cur, ldh, g, ldx, M, precision);
    a.res = g; a.ldres = ldx;
    rc = fc_launch_gemm(a, s);
    if (rc || !attn) return rc;
    rc = fc_launch_gemm(fc_gemm_linear(gl.cpl.in_o, cur, ldh, gw.dO, 64, M, precision), s);
    if (rc) return rc;
    return attn_backward(f, pre, gl, B, N, Nc, gw, g, ldx, precision, s, sgrad, sgrad_add, cap);
}

// cap: the attention blocks whose score gradients are written (fc_flow_attention_score_grads); the walk meets them in
// decreasing slot order, layers L-1 ... 0 then the augmenter
static int flow_log_prob_grad(const fc_flow* f, const float* x, const float* context, const float* extra, const float* eps,
                              float* log_prob_out, float* grad_out, int B, int N, int Nc, void* workspace, int64_t workspace_bytes,
                              int precision, fc_stream_t stream_, const FcCapture* cap = nullptr) {
    FC_REQUIRE(f && x && context && log_prob_out && grad_out && B > 0 && N > 0 && Nc > 0);
    if (f->cpl_kind != FC_CPL_AFFINE || f->cif_dim) return FC_ERR_UNSUPPORTED;
    if (!f->glayers) return FC_ERR_MODEL;
    FC_REQUIRE((int64_t)B * N <= FC_GRAD_MAX_ROWS);
    FC_REQUIRE(eps || !f->has_aug);
    GradWs gw = carve_grad_ws(f, B, N, Nc, workspace);
    if (!ws_ok(workspace, gw.total_bytes, workspace_bytes)) return FC_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream_;
    int rc = flow_forward(f, x, context, extra, eps, nullptr, log_prob_out, nullptr, B, N, Nc, workspace, gw.fw.total_bytes, precision,
                          stream_, nullptr, 0, gw.ckpt);
    if (rc) return rc;
    const int M = B * N, ldx = gw.fw.ldx;
    auto slot = [&](int l) { return gw.ckpt + (size_t)l * M * ldx; };
    // the base density N(0, I): d/dz sum(-z^2/2) = -z; ActNorm and LinearLU log-dets are constants
    float* g = gw.gA; float* g_other = gw.gB;
    rc = fc_launch_neg_copy(slot(f->L), ldx, g, ldx, M, f->D, s);
    if (rc) return rc;
    int n_captured = 0;
    bool sgrad_add = false;
    auto sgrad_for = [&](int cslot) -> float* {
        if (!cap || n_captured >= cap->n_slots || cap->slots[cap->n_slots - 1 - n_captured] != cslot) return nullptr;
        const size_t i = cap->accumulate ? 0 : (size_t)(cap->n_slots - 1 - n_captured);
        sgrad_add = cap->accumulate && n_captured > 0;       // the first block met stores, the later ones add
        ++n_captured;
        return cap->out + i * (size_t)B * (size_t)cap->n_query * (size_t)Nc;
    };
    for (int l = f->L - 1; l >= 0; --l) {
        const FcFlowLayer& y = f->layers[l];
        const FcGradLayer& gl = f->glayers[l];
        if (y.has_lu) {
            // dz = g (W' - diag) + diag * g: the forward's off-diagonal / diagonal split, transposed
            rc = lu_gemm(gl.lu, y.lu_diag, g, g_other, ldx, M, precision, s);
            if (rc) return rc;
            float* t = g; g = g_other; g_other = t;
        }
        float* sg = sgrad_for(l + 1);
        rc = conditioner_backward(f, y.pre, y.attn, y.cpl, gl, false, slot(l), l + 1, context, nullptr, B, N, Nc, gw, g, precision, s,
                                  sg, sgrad_add, cap);
        if (rc) return rc;
    }
    if (f->has_aug) {
        float* sg = sgrad_for(0);
        rc = conditioner_backward(f, f->augpre, f->augattn, f->aug, f->gaug, true, slot(0), 0, context, eps, B, N, Nc, gw, g,
                                  precision, s, sg, sgrad_add, cap);
        if (rc) return rc;
    }
    return copy_cols(g, ldx, grad_out, f->d_in, M, f->d_in, s);
}

extern "C" int fc_flow_log_prob_grad(const fc_flow* f, const float* x, const float* context, const float* extra, const float* eps,
                                     float* log_prob_out, float* grad_out, int B, int N, int Nc, void* workspace,
                                     int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    return flow_log_prob_grad(f, x, context, extra, eps, log_prob_out, grad_out, B, N, Nc, workspace, workspace_bytes, precision,
                              stream_);
}

// The input-gradient pass that also writes d lp_i / d s_ij of the attention blocks listed in slots_host (see FcCapture), read at
// the start of each captured block's attention backward.  Only reads are added, so log_prob and grad are fc_flow_log_prob_grad's.
extern "C" int fc_flow_attention_score_grads(const fc_flow* f, const float* x, const float* context, const float* extra,
                                             const float* eps, const int32_t* slots_host, int n_slots, const int32_t* query_idx,
                                             int n_query, int accumulate, float* maps_out, float* log_prob_out, float* grad_out,
                                             int B, int N, int Nc, void* workspace, int64_t workspace_bytes, int precision,
                                             fc_stream_t stream_) {
    FC_REQUIRE(f && slots_host && n_slots > 0 && maps_out && n_query > 0);
    if (f->is_global) return FC_ERR_UNSUPPORTED;       // no attention over context points: the device never runs one
    if (f->cpl_kind != FC_CPL_AFFINE || f->cif_dim) return FC_ERR_UNSUPPORTED;
    if (!f->glayers) return FC_ERR_MODEL;
    FC_REQUIRE(query_idx || n_query == N);
    for (int i = 0; i < n_slots; ++i)
        FC_REQUIRE(slots_host[i] >= 0 && slots_host[i] <= f->L && (i == 0 || slots_host[i] > slots_host[i - 1]));
    FC_REQUIRE(slots_host[0] != 0 || f->has_aug);     // an identity augmenter has no attention
    const FcCapture cap{slots_host, n_slots, query_idx, n_query, maps_out, accumulate != 0};
    return flow_log_prob_grad(f, x, context, extra, eps, log_prob_out, grad_out, B, N, Nc, workspace, workspace_bytes, precision,
                              stream_, &cap);
}
