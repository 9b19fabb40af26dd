// fp32 GEMM with fused epilogues -- the contraction workhorse of the path
// (reference: every nn.Linear / 1x1 conv on the path, SURVEY.md 2.2 F3-F8).
#pragma once
#include "common.cuh"

enum { FC_ACT_NONE = 0, FC_ACT_GELU = 1, FC_ACT_LRELU = 2, FC_ACT_RELU = 3 };

// Epilogue kinds.  All operate on the fp32 accumulator tile while it is still in registers, so the
// elementwise tail of each reference op never makes a separate trip through HBM.
enum {
    FC_EPI_STORE = 0,     // C = act(acc + bias (+ res))
    FC_EPI_LNQ = 1,       // C = rstd[row]*(acc - mu[row]*csum[n]) + bias[n]   (LayerNorm folded into to_q)
    FC_EPI_COUPLING = 2,  // affine coupling: columns interleaved (s_raw_j, t_j); x2 updated in place; ldj partial
    FC_EPI_AUGMENT = 3,   // augment: columns interleaved (mean_j, log_std_j); z2 written; ldj partial
    FC_EPI_KVSPLIT = 4,   // to_kv for the tcgen05 attention (N = 128): k -> TF32 hi/lo [M][64]; v -> hi/lo TRANSPOSED
                          // per cloud [B][64][kv_ncp]  (tcgen05 path only)
    FC_EPI_COUPLING_INV = 5,  // inverse affine coupling (sampling pass): x2 = (y2 - t) / s in place, no log-det
};

struct GemmArgs {
    // A is the concatenation [A1 (K1 cols) | A2 (K2 cols)] along K; A2 may be null (K2 = 0).
    const float* A1; int lda1; int K1;
    const float* A2; int lda2; int K2;
    // Wt: K-major weights [Kp1 + Kp2][ldw], Kp = K rounded up to 16 (padding rows are zero).
    const float* Wt; int ldw;
    // bias[n] if bias_group == 0, else bias[(row / bias_group) * bias_ld + n]  (per-cloud bias)
    const float* bias; int bias_ld; int bias_group;
    const float* res; int ldres;   // optional residual added before the activation
    const float* res_scale;        // optional per-column factor on the residual (the LinearLU diagonal)
    int act;
    float* C; int ldc;
    int M, N;
    int epi;
    // FC_EPI_LNQ
    const float* row_mu; const float* row_rstd; const float* csum;
    // FC_EPI_COUPLING / FC_EPI_AUGMENT: x is the latent buffer [M][ldx]; the updated half starts at col0
    float* x; int ldx; int col0;
    float* part;                   // [gridDim.x][M] partial log-det sums (deterministic, no atomics)
    const float* eps; int ld_eps;  // FC_EPI_AUGMENT
    // FC_EPI_KVSPLIT: C = k hi (ldc = 64), kv_klo = k lo; v^T hi / lo; rows are (cloud, key) = (row / kv_nc, row % kv_nc)
    float* kv_klo; float* kv_vthi; float* kv_vtlo; int kv_nc; int kv_ncp;
    int kv_f16;                    // 0: TF32 hi/lo stored as fp32; 1: the four outputs are fp16 hi / fp16 (x - hi) (kv_ncp in halfs)
    int precision;                 // 0 fp32 FFMA, 1 3xTF32 tcgen05 (where available)
    // tcgen05 path: the same weight pre-split into TF32 hi / lo parts, N-major rows, K contiguous:
    // [n_tiles*BN][ldk] with ldk = round32(K1) + round32(K2) (zero padded); null -> FFMA only
    const float* Whi; const float* Wlo; int ldk;
    // format of Whi / Wlo: 0 = TF32 hi / lo parts stored as fp32 (3xTF32 kernel); 1 = fp16 hi and fp16 (W - hi) * 2^11
    // (3xFP16 kernel: same 11-bit significands, twice the tensor rate and half the operand bytes; see gemm_tc.cu)
    int tc_fmt;
};

// tcgen05 tiling of the N dimension: n_tiles = ceil(N/96), BN = ceil(N/n_tiles) rounded up to 16.
// BN <= 96: two double-buffered accumulators (main + compensation) take 384 of the 512 TMEM columns, the A operand the rest.
static inline int fc_tc_n_tiles(int N) { return (N + 95) / 96; }
static inline int fc_tc_bn(int N) { const int t = fc_tc_n_tiles(N); return fc_round_up((N + t - 1) / t, 16); }
static inline int fc_tc_kpad(int K) { return fc_round_up(K, 32); }

static inline GemmArgs fc_gemm_args_zero() {
    GemmArgs a;
    a.A1 = nullptr; a.lda1 = 0; a.K1 = 0; a.A2 = nullptr; a.lda2 = 0; a.K2 = 0;
    a.Wt = nullptr; a.ldw = 0; a.bias = nullptr; a.bias_ld = 0; a.bias_group = 0;
    a.res = nullptr; a.ldres = 0; a.res_scale = nullptr; a.act = FC_ACT_NONE; a.C = nullptr; a.ldc = 0; a.M = 0; a.N = 0;
    a.epi = FC_EPI_STORE; a.row_mu = nullptr; a.row_rstd = nullptr; a.csum = nullptr;
    a.x = nullptr; a.ldx = 0; a.col0 = 0; a.part = nullptr; a.eps = nullptr; a.ld_eps = 0;
    a.kv_klo = nullptr; a.kv_vthi = nullptr; a.kv_vtlo = nullptr; a.kv_nc = 0; a.kv_ncp = 0; a.kv_f16 = 0;
    a.precision = 0; a.Whi = nullptr; a.Wlo = nullptr; a.ldk = 0; a.tc_fmt = 0;
    return a;
}

// Number of N-tiles (== number of partial-sum slabs an epilogue with `part` writes).
int fc_gemm_n_tiles(int N);
// ldw the packer must use for an N-column weight.
static inline int fc_gemm_ldw(int N) { return N <= 64 ? 64 : fc_round_up(N, 128); }
static inline int fc_gemm_kpad(int K) { return fc_round_up(K, 16); }

int fc_launch_gemm(const GemmArgs& a, cudaStream_t stream);       // dispatches on a.precision
int fc_launch_gemm_ffma(const GemmArgs& a, cudaStream_t stream);  // exact fp32 path

void fc_count_launch(int n = 1);
