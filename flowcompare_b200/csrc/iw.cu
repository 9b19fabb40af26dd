// Multi-draw log-likelihood (fc_flow_log_prob_draws, fc_logmeanexp): the importance-weighted estimate
//   IW_K(x) = log( (1/K) * sum_k exp(lp_k) )
// over K augmentation draws lp_k of `Flow.log_prob` (reference models/augmenter.py:49-63: each draw's exp(lp_k) is an unbiased
// estimate of p(x | c)), and the row interleave the K-draw forward pass uses.
#include "model.cuh"

namespace {

// Draw k's augmented latent, staged as rows r = b*N + n, and its partial log-det slabs [n_part][M0] -> row (b*K + k)*N + n of
// the K-draw layout (latent dst [M0*K][ldd], slabs part_dst [n_part][M0*K]).  One thread per copied float.
__global__ void scatter_draw_kernel(const float* __restrict__ src, int lds, int cols, const float* __restrict__ part_src,
                                    int n_part, float* __restrict__ dst, int ldd, float* __restrict__ part_dst, int N, int K,
                                    int k, long long M0) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int W = cols + n_part;
    if (i >= M0 * W) return;
    const long long r = i / W;
    const int c = (int)(i % W);
    const long long rd = (r / N * K + k) * N + r % N;
    if (c < cols) dst[rd * ldd + c] = src[r * lds + c];
    else part_dst[(c - cols) * (M0 * K) + rd] = part_src[(c - cols) * M0 + r];
}

// out[i] = m + (log(sum_k exp(draws[k][i] - m)) - log K), m = max_k draws[k][i]; one thread per point, the draws folded in
// index order in fp32, so the value depends on nothing but the point's own K draws.  NaN if any draw is NaN, +inf if any is
// +inf, -inf draws add exp(-inf) = 0 (all -inf: -inf).  K equal finite draws give that value exactly: the sum is K, and
// log(K) - log(K) is 0 before it is added to m.
__global__ void logmeanexp_kernel(const float* __restrict__ draws, int K, long long M, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    float m = -INFINITY;
    bool nan = false;
    for (int k = 0; k < K; ++k) {
        const float v = draws[k * M + i];
        nan |= (v != v);
        m = fmaxf(m, v);              // fmaxf ignores a NaN operand: tracked separately
    }
    if (nan) { out[i] = NAN; return; }
    if (!(m > -INFINITY && m < INFINITY)) { out[i] = m; return; }
    float s = 0.f;
    for (int k = 0; k < K; ++k) s += expf(draws[k * M + i] - m);
    out[i] = m + (logf(s) - logf((float)K));
}

}  // namespace

int fc_launch_scatter_draw(const float* src, int lds, int cols, const float* part_src, int n_part, float* dst, int ldd,
                           float* part_dst, int B, int N, int K, int k, cudaStream_t s) {
    FC_REQUIRE(src && dst && cols > 0 && (n_part == 0 || (part_src && part_dst)) && B > 0 && N > 0 && k >= 0 && k < K);
    const long long M0 = (long long)B * N, tot = M0 * (cols + n_part);
    scatter_draw_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(src, lds, cols, part_src, n_part, dst, ldd, part_dst, N, K,
                                                                      k, M0);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

extern "C" int fc_logmeanexp(const float* draws, int K, int64_t M, float* out, fc_stream_t stream) {
    FC_REQUIRE(draws && out && K > 0 && M > 0);
    logmeanexp_kernel<<<(unsigned)((M + 255) / 256), 256, 0, (cudaStream_t)stream>>>(draws, K, (long long)M, out);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}
