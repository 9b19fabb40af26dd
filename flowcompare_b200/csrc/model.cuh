// Packed-model descriptions shared by flow.cu / embed.cu / api.cu.
// Arena format: see DESIGN.md "arena format" and flowcompare_b200/packing.py (the two walk the
// tensors in the same order; the table is a flat list of float offsets into the arena).
#pragma once
#include "common.cuh"
#include "gemm.cuh"

constexpr int FC_MAX_HIDDEN = 8;
constexpr int32_t FC_FLOW_MAGIC = 0x46435F46;  // 'FC_F'
constexpr int32_t FC_EMB_MAGIC = 0x46435F45;   // 'FC_E'
constexpr int32_t FC_INV_MAGIC = 0x46435F49;   // 'FC_I': inverse ActNorm+LinearLU matrices of the sampling pass
constexpr int32_t FC_GRAD_MAGIC = 0x46435F47; // 'FC_G': transposed weights of the input-gradient pass
constexpr int32_t FC_ARENA_VERSION = 2;       // tensor-core weight copies: TF32 hi/lo (fp32 storage)
constexpr int32_t FC_ARENA_VERSION_F16 = 3;    // tensor-core weight copies: fp16 hi / scaled lo

struct FcLinear {
    const float* w = nullptr;  // K-major [Kp][ldw]
    const float* b = nullptr;  // [N] or null
    const float* whi = nullptr; const float* wlo = nullptr;  // tcgen05 copies [n_tiles*BN][ldk] or null
    int K1 = 0, K2 = 0, N = 0, ldw = 0, ldk = 0;
    int tc_fmt = 0;            // format of whi / wlo (GemmArgs::tc_fmt)
};

// C = A1 l + l.b through the plain-store epilogue: every field of the packed Linear (K1, K2, N, its bias, the FFMA weights, the
// tensor-core copies, their K stride and format) is bound here, so no caller can drop one and silently take another GEMM path
// or format.  Callers set only what differs: A2 / lda2, a bias override, res / res_scale, act and the epilogue fields.
static inline GemmArgs fc_gemm_linear(const FcLinear& l, const float* A1, int lda1, float* C, int ldc, int M, int precision) {
    GemmArgs g = fc_gemm_args_zero();
    g.A1 = A1; g.lda1 = lda1; g.K1 = l.K1; g.K2 = l.K2; g.N = l.N; g.bias = l.b;
    g.Wt = l.w; g.ldw = l.ldw; g.Whi = l.whi; g.Wlo = l.wlo; g.ldk = l.ldk; g.tc_fmt = l.tc_fmt;
    g.C = C; g.ldc = ldc; g.M = M; g.precision = precision;
    return g;
}

struct FcMlp {
    FcLinear in;
    FcLinear hidden[FC_MAX_HIDDEN];
    int n_hidden = 0;
    FcLinear out;
    int act = FC_ACT_GELU;   // non-linearity of the in / hidden layers (reference models/nets.py:10)
};

struct FcAttn {
    const float* csum = nullptr;   // [inner] column sums of Wq*diag(gamma)
    const float* qbias = nullptr;  // [inner] Wq*beta
    FcLinear q;                    // K=attn_in -> inner
    FcLinear kv;                   // K=E -> 2*inner
};

struct FcFlowLayer {
    FcMlp pre;      // pre-attention MLP (attention configs)
    FcAttn attn;
    FcMlp cpl;      // coupling conditioner; in.K2 = inner for attention configs
    FcLinear lu;    // folded ActNorm + LinearLU minus its diagonal (absent on the last layer)
    const float* lu_diag = nullptr;  // [D] the diagonal, applied to the latent in the GEMM epilogue
    bool has_lu = false;
    // sampling pass (fc_flow_set_inverse): (ActNorm + LinearLU)^-1 = Wp^-1 z' + shift, same diagonal / off-diagonal split
    FcLinear lu_inv;
    const float* lu_inv_diag = nullptr;
    // exponential coupling: the four squashing scalars (scale, shift, rescale, reshift; models/exponential_coupling.py:22-25)
    const float* expo_sq = nullptr;
    // CIF block (models/cif_block.py:50-68): the ConditionalNormal net shared by the augmenter and the slicer, the affine
    // coupling that conditions x on the augmented part (both Reverse permutations folded into its weights), and the
    // ActNorm between them as one per-column affine map over the cif_dim columns
    FcMlp cifnet, affcif;
    const float* cif_sc = nullptr; const float* cif_bi = nullptr;
    const float* cif_isc = nullptr; const float* cif_ibi = nullptr;   // its inverse (sampling pass, fc_flow_set_inverse)
};

// Transposed weights of the input-gradient pass (fc_flow_set_grad; flow_grad.cu).  Every backward contraction dX = dY W is a
// Linear whose weight is W^T: `in_x` / `in_o` are the first layer's x columns and attention-output columns (the latter with the
// out-projection folded in), hidden[i] / out the transposes of the forward's layers of the same index.
struct FcMlpT { FcLinear in_x, in_o; FcLinear hidden[FC_MAX_HIDDEN]; FcLinear out; };
struct FcGradLayer { FcMlpT pre, cpl; FcLinear q, lu; };   // q: Wq diag(gamma) transposed; lu: the off-diagonal part transposed

struct fc_flow {
    int L, D, d_in, half, extra, is_global, E, inner, attn_in, hid, n_hid, pre_hid, n_pre_hid,
        aug_hid, n_aug_hid, augpre_hid, n_augpre_hid;
    double ldj_const;            // sum over layers of ActNorm + LinearLU log-dets (exact, fp64 at pack time)
    FcMlp augpre;
    FcAttn augattn;
    FcMlp aug;
    bool has_cb = false;
    FcLinear cb;                 // per-cloud bias GEMM: K = extra + (global ? E : 0), N = (L+1)*hid
    FcFlowLayer* layers = nullptr;
    const float* arena = nullptr;
    int64_t arena_floats = 0;
    bool has_inverse = false;    // fc_flow_set_inverse was called (needed by fc_flow_sample)
    FcGradLayer* glayers = nullptr;   // fc_flow_set_grad: per coupling layer, and the augmenter's in `gaug`
    FcGradLayer gaug;
    // transforms no shipped config builds (SURVEY.md 8 a18; header words 19..): coupling kind 0 affine / 1 rational-quadratic
    // spline / 2 exponential, conditioner non-linearity, identity augmenter (latent_dim == input_dim), CIF block
    int cpl_kind = 0, num_bins = 0, act = FC_ACT_GELU, has_aug = 1;
    int cif_dim = 0, cif_hid = 0, n_cif_hid = 0, affcif_hid = 0, n_affcif_hid = 0;
    float cif_clamp = 0.f;
};
enum { FC_CPL_AFFINE = 0, FC_CPL_SPLINE = 1, FC_CPL_EXPO = 2 };

struct FcEdgeConv { FcLinear pq; int Cin, Cout; };

struct fc_embedder {
    int kind;        // 0 DGCNN per-point, 1 DGCNN global, 2 PAConv
    int d_in, k, E, out_hid, n_out_hid;
    FcEdgeConv ec[4];
    FcLinear conv5;
    FcMlp out_mlp;
    void* paconv = nullptr;  // PAConv description (paconv.cu)
    const float* arena = nullptr;
    int64_t arena_floats = 0;
};

// table cursor used by the *_create functions
struct FcCursor {
    const int64_t* table; int n; int pos; const float* arena; int64_t arena_floats; bool ok;
    int tc_fmt = 0;
    int64_t next() { if (pos >= n) { ok = false; return -1; } return table[pos++]; }
    const float* ptr(int64_t off, int64_t count) {
        if (off < 0) return nullptr;
        if (off + count > arena_floats || (off & 3)) { ok = false; return nullptr; }
        return arena + off;
    }
    FcLinear linear(int K1, int K2, int N, bool has_bias = true) {
        FcLinear l; l.K1 = K1; l.K2 = K2; l.N = N; l.ldw = fc_gemm_ldw(N);
        const int64_t kp = fc_gemm_kpad(K1) + (K2 ? fc_gemm_kpad(K2) : 0);
        l.w = ptr(next(), kp * l.ldw);
        const int64_t boff = next();
        l.b = has_bias ? ptr(boff, N) : nullptr;
        if (!l.w || (has_bias && !l.b)) ok = false;
        const int64_t hoff = next(), loff = next();
        if (hoff >= 0 && loff >= 0) {
            l.ldk = fc_tc_kpad(K1) + (K2 ? fc_tc_kpad(K2) : 0);
            const int64_t cnt = (int64_t)fc_tc_n_tiles(N) * fc_tc_bn(N) * l.ldk / (tc_fmt ? 2 : 1);   // fp16: two per float slot
            l.whi = ptr(hoff, cnt); l.wlo = ptr(loff, cnt); l.tc_fmt = tc_fmt;
            if (!l.whi || !l.wlo) ok = false;
        }
        return l;
    }
    FcMlp mlp(int K1, int K2, int hid, int n_hidden, int N_out) {
        FcMlp m; m.n_hidden = n_hidden;
        if (n_hidden > FC_MAX_HIDDEN) { ok = false; return m; }
        m.in = linear(K1, K2, hid);
        for (int i = 0; i < n_hidden; ++i) m.hidden[i] = linear(hid, 0, hid);
        m.out = linear(hid, 0, N_out);
        return m;
    }
};

// misc kernels (flow.cu)
int fc_launch_ln_stats(const float* h, int ldh, int M, int width, float eps, float* mu, float* rstd, cudaStream_t s);
int fc_launch_cross_attention(const float* q, int ldq, const float* kv, int ldkv, float* out, int ldo,
                              int B, int N, int Nc, int d, float scale, cudaStream_t stream);
// tcgen05 / TMEM version (attention_tc.cu); scratch holds the TF32 hi/lo copies of k and v^T
int64_t fc_attention_tc_scratch_floats(int B, int Nc);
void fc_attention_tc_scratch_layout(int B, int Nc, float* scratch, float** khi, float** klo, float** vthi, float** vtlo,
                                    int* ncp, int fmt);
int fc_launch_cross_attention_tc(const float* q, int ldq, const float* kv, int ldkv, float* out, int ldo, int B, int N,
                                 int Nc, int d, float scale, float* scratch, int presplit, int fmt, cudaStream_t stream);
// the softmax weights of one attention block, P [B, n_query, Nc] (attention_maps.cu); qidx: device list of query rows or null
int fc_launch_attention_maps(const float* q, int ldq, const float* kv, int ldkv, const int32_t* qidx, int n_query,
                             float* out, int B, int N, int Nc, float scale, cudaStream_t stream);
int fc_launch_edgeconv_gather_max(const float* PQ, int ldpq, const int32_t* idx, int B, int N, int k, int Cout,
                                  float* out, int ldo, cudaStream_t stream);
int fc_knn_launch(const float* q, int ldq, long long q_bstride, const float* t, int ldt, long long t_bstride,
                  int B, int Nq, int Nt, int C, int k, int mode, int32_t* idx32, int64_t* idx64, float* norms_scratch,
                  cudaStream_t stream);
int64_t fc_knn_scratch_floats(int B, int Nq, int Nt, bool self);   // floats of `norms_scratch` (squared norms of the points)

// elementwise tails of the spline / exponential couplings and the CIF block (transforms.cu)
int fc_launch_rq_spline(const float* params, int ldp, float* lat, int ldx, int col0, int n2, int nb, int M, float* part,
                        int inverse, cudaStream_t s);
int fc_launch_cond_normal(const float* params, int ldp, float* lat, int ldx, int col0, int S, const float* eps, int M,
                          float clamp, float* part, int mode, cudaStream_t s);
int fc_launch_col_affine(float* lat, int ldx, int cols, long long M, const float* sc, const float* bi, cudaStream_t s);
int fc_launch_expm_action(const float* params, int ldp, float* lat, int ldx, int col0, int n2, const float* squash4,
                          float* part, long long row0, int rows, int inverse, cudaStream_t s);
int fc_expm_max_n();

// K-draw forward (iw.cu): copies draw k's staged latent columns [0, cols) and log-det slabs, rows b*N + n, to rows
// (b*K + k)*N + n of the K-draw layout
int fc_launch_scatter_draw(const float* src, int lds, int cols, const float* part_src, int n_part, float* dst, int ldd,
                           float* part_dst, int B, int N, int K, int k, cudaStream_t s);
constexpr int64_t FC_DRAWS_MAX_ROWS = 1ll << 20;   // rows of one fc_flow_log_prob_draws pass

// input-gradient pass (flow_grad.cu)
int fc_launch_act_fwd(const float* pre, int ldp, float* post, int ldq, long long M, int width, int act, int fast, cudaStream_t s);
int fc_launch_act_bwd(float* d, int ldd, const float* pre, int ldp, long long M, int width, int act, cudaStream_t s);
int fc_launch_coupling_tail_bwd(const float* raw, int ldr, const float* x, int ldx, float* g, int ldg, int col0, int n2, float* dst,
                                int ldd, int M, cudaStream_t s);
int fc_launch_augment_tail_bwd(const float* raw, int ldr, const float* eps, int S, const float* g, int ldg, int col0, float* dst,
                               int ldd, int M, cudaStream_t s);
int fc_launch_ln_bwd(const float* h, int ldh, const float* mu, const float* rstd, float* d, int ldd, int M, int width, cudaStream_t s);
int fc_launch_neg_copy(const float* z, int ldz, float* g, int ldg, long long M, int cols, cudaStream_t s);
int fc_launch_attention_dq(const float* q, const float* kv, int ldkv, const float* o, const float* dO, float* dq, int B, int N,
                           int Nc, float scale, cudaStream_t stream);
constexpr int64_t FC_GRAD_MAX_ROWS = 1ll << 16;   // rows of one fc_flow_log_prob_grad pass
bool fc_gemm_tc_supported(const GemmArgs& a);      // gemm_tc.cu

// runs in/hidden layers of an MLP; returns the buffer holding the last hidden activation.
// bufA/bufB: [M][ldh] scratch (ldh >= hidden width).  `in_bias`/group override the in-layer bias.
struct FcMlpIn {
    const float* A1; int lda1; const float* A2; int lda2;
    const float* bias; int bias_ld; int bias_group;  // bias == nullptr -> use the packed in-layer bias
};
int fc_run_mlp_hidden(const FcMlp& m, const FcMlpIn& in, int M, float* bufA, float* bufB, int ldh,
                      int precision, cudaStream_t stream, float** last);
