// Elementwise and attention kernels of the input-gradient pass (fc_flow_log_prob_grad, driver in flow.cu): the backward of
// everything on the flow's path that is not a GEMM.  Every backward contraction dX = dY W runs on the existing GEMM kernels with
// the transposed weights of packing.pack_flow_grad; what is left is
//   - the conditioners' non-linearities: the recompute stores pre-activations and applies the forward's own device GELU (the
//     exact erf form on the FFMA path, fc_gelu_erf_fast on the tcgen05 path), the backward multiplies by the exact derivative;
//   - the affine coupling's tail (reference models/affine_coupling.py:40-46) and the augmenter's (models/augmenter.py:49-63);
//   - LayerNorm (models/perceiver.py:26-35) and the attention's dQ (perceiver.py:108-115).
// Everything is fp32, each output computed from its own row in a fixed order: deterministic and independent of the batch.
#include <atomic>
#include "model.cuh"

namespace {

// post = act(pre): the forward's activation of the GEMM path that produced `pre` (fast: the tcgen05 epilogue's GELU)
__global__ void act_fwd_kernel(const float* __restrict__ pre, int ldp, float* __restrict__ post, int ldq, long long M, int width,
                               int act, int fast) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * width) return;
    const long long r = i / width; const int c = (int)(i % width);
    const float x = pre[r * ldp + c];
    float y = x;
    if (act == FC_ACT_GELU) y = fast ? fc_gelu_erf_fast(x) : fc_gelu_erf(x);
    else if (act == FC_ACT_RELU) y = fmaxf(x, 0.f);
    post[r * ldq + c] = y;
}

// d <- d * act'(pre): GELU' = Phi(x) + x phi(x) (exact), ReLU' = [x > 0]
__global__ void act_bwd_kernel(float* __restrict__ d, int ldd, const float* __restrict__ pre, int ldp, long long M, int width,
                               int act) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * width) return;
    const long long r = i / width; const int c = (int)(i % width);
    const float x = pre[r * ldp + c];
    float g;
    if (act == FC_ACT_GELU)
        g = fmaf(x, 0.39894228040143267794f * expf(-0.5f * x * x), 0.5f * (1.0f + erff(x * 0.70710678118654752440f)));
    else
        g = x > 0.f ? 1.f : 0.f;
    d[r * ldd + c] *= g;
}

// Affine coupling, s = 2 sigmoid(a) (what FC_EPI_COUPLING evaluates), y2 = x2 s + t, log s added to the objective.  raw: the
// conditioner's interleaved (a_j, t_j) outputs; x2 = x[:, col0 + j] the layer's input; g[:, col0 + j] = dL/dy2 on entry.
//   dst = (d_a, d_t) interleaved = ((g y2 x2 s + 1)(1 - s/2), g_y2);  g[:, col0 + j] <- g_y2 s
__global__ void coupling_tail_bwd_kernel(const float* __restrict__ raw, int ldr, const float* __restrict__ x, int ldx,
                                         float* __restrict__ g, int ldg, int col0, int n2, float* __restrict__ dst, int ldd, int M) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * n2) return;
    const long long r = i / n2; const int j = (int)(i % n2);
    const float a = raw[r * ldr + 2 * j];
    const float sig = 1.0f / (1.0f + expf(-a));
    const float s = (2.0f * sig - 1.0f) + 1.0f;
    const float gy = g[r * ldg + col0 + j];
    const float x2 = x[r * ldx + col0 + j];
    dst[r * ldd + 2 * j] = fmaf(gy * x2, s, 1.0f) * (1.0f - 0.5f * s);
    dst[r * ldd + 2 * j + 1] = gy;
    g[r * ldg + col0 + j] = gy * s;
}

// Augmenter, e = mean + exp(ls) eps, +ls added to the objective (FC_EPI_AUGMENT).  raw: interleaved (mean_j, ls_j); g[:, col0 + j]
// = dL/de.  dst = (d_mean, d_ls) = (g_e, g_e exp(ls) eps + 1)
__global__ void augment_tail_bwd_kernel(const float* __restrict__ raw, int ldr, const float* __restrict__ eps, int S,
                                        const float* __restrict__ g, int ldg, int col0, float* __restrict__ dst, int ldd, int M) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)M * S) return;
    const long long r = i / S; const int j = (int)(i % S);
    const float ls = raw[r * ldr + 2 * j + 1];
    const float ge = g[r * ldg + col0 + j];
    dst[r * ldd + 2 * j] = ge;
    dst[r * ldd + 2 * j + 1] = fmaf(ge * expf(ls), eps[r * S + j], 1.0f);
}

// LayerNorm backward (no affine: the gain is folded into the transposed to_q), one warp per row, in place on d:
// dh = rstd (dxh - mean(dxh) - xh mean(dxh xh)),  xh = (h - mu) rstd
__global__ void ln_bwd_kernel(const float* __restrict__ h, int ldh, const float* __restrict__ mu, const float* __restrict__ rstd,
                              float* __restrict__ d, int ldd, int M, int width) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= M) return;
    const float m = mu[row], rs = rstd[row];
    const float* hp = h + (size_t)row * ldh;
    float* dp = d + (size_t)row * ldd;
    float xh[16], dx[16];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int c = i * 32 + lane;
        xh[i] = 0.f; dx[i] = 0.f;
        if (c < width) { xh[i] = (hp[c] - m) * rs; dx[i] = dp[c]; s1 += dx[i]; s2 = fmaf(dx[i], xh[i], s2); }
    }
    s1 = fc_warp_sum(s1) / (float)width;
    s2 = fc_warp_sum(s2) / (float)width;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int c = i * 32 + lane;
        if (c < width) dp[c] = rs * (dx[i] - s1 - xh[i] * s2);
    }
}

__global__ void neg_copy_kernel(const float* __restrict__ z, int ldz, float* __restrict__ g, int ldg, long long M, int cols) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * cols) return;
    const long long r = i / cols; const int c = (int)(i % cols);
    g[r * ldg + c] = -z[r * ldz + c];
}

// ------------------------------------------------------------------------------------------------ attention dQ
// o = softmax(q k^T scale) v  =>  dq_i = scale sum_j P_ij (dO_i . v_j - D_i) k_j,  D_i = dO_i . o_i,  P recomputed.
// Modelled on attention_maps_kernel: CTA = 128 query rows of one cloud, 128 threads, 8 x 8 register tiles (rows tq*4.. and
// 64+tq*4.., keys / head dims tk*4.. and 32+tk*4..), keys streamed through shared memory in 64-key tiles twice: pass 1 keeps the
// online row max and sum, pass 2 recomputes the scores, forms W_ij = P_ij (dp_ij - D_i) into shared memory and accumulates
// dq += W k.  Every dot product and the dq accumulation are sequential fp32 FMA chains in a fixed order (d, then keys in index
// order), so a row's dq depends on its own row and the cloud's keys only.
constexpr int GD = 64, GQ = 128, GK = 64, GTHREADS = 128;
constexpr int GQLD = GQ + 4, GKLD = GK + 4, GDLD = GD + 4;

struct DqSmem {
    float Qt[GD][GQLD];    // q transposed [d][row]
    float Gt[GD][GQLD];    // dO transposed
    float Kt[GD][GKLD];    // k transposed [d][key]
    float Vt[GD][GKLD];    // v transposed
    float Kr[GK][GDLD];    // k [key][d]
    float Wt[GK][GQLD];    // W [key][row]
    float Dr[GQ];          // D_i
    float Mr[GQ], Lr[GQ];  // row max of the scaled scores, 1 / row sum of exp (pass 1)
};

__device__ __forceinline__ int g_col(int t, int j) { return (j < 4 ? t * 4 : 32 + t * 4) + (j & 3); }
__device__ __forceinline__ int g_row(int tq, int i) { return i < 4 ? tq * 4 + i : 64 + tq * 4 + (i - 4); }

__global__ void __launch_bounds__(GTHREADS, 1) attention_dq_kernel(const float* __restrict__ q, const float* __restrict__ kv,
                                                                    int ldkv, const float* __restrict__ o,
                                                                    const float* __restrict__ dO, float* __restrict__ dq, int N,
                                                                    int Nc, float scale) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DqSmem& sm = *reinterpret_cast<DqSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int tk = tid & 7, tq = tid >> 3;
    const int b = blockIdx.y;
    const int r0 = blockIdx.x * GQ;
    const size_t qb = (size_t)b * N;
    const float* kb = kv + (size_t)b * Nc * ldkv;

    for (int e = tid; e < GQ * (GD / 4); e += GTHREADS) {
        const int r = e / (GD / 4), c4 = (e % (GD / 4)) * 4;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), c = a;
        if (r0 + r < N) {
            a = *reinterpret_cast<const float4*>(q + (qb + r0 + r) * GD + c4);
            c = *reinterpret_cast<const float4*>(dO + (qb + r0 + r) * GD + c4);
        }
        sm.Qt[c4 + 0][r] = a.x; sm.Qt[c4 + 1][r] = a.y; sm.Qt[c4 + 2][r] = a.z; sm.Qt[c4 + 3][r] = a.w;
        sm.Gt[c4 + 0][r] = c.x; sm.Gt[c4 + 1][r] = c.y; sm.Gt[c4 + 2][r] = c.z; sm.Gt[c4 + 3][r] = c.w;
    }
    {   // D_i = dO_i . o_i, one row per thread
        float dd = 0.f;
        if (r0 + tid < N) {
            const float* op = o + (qb + r0 + tid) * GD;
            const float* gp = dO + (qb + r0 + tid) * GD;
            for (int d = 0; d < GD; ++d) dd = fmaf(gp[d], op[d], dd);
        }
        sm.Dr[tid] = dd;
    }
    auto stage_keys = [&](int k0, bool all) {
        __syncthreads();
        for (int e = tid; e < GK * (GD / 4); e += GTHREADS) {
            const int r = e / (GD / 4), c4 = (e % (GD / 4)) * 4;
            float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
            if (k0 + r < Nc) {
                kk = *reinterpret_cast<const float4*>(kb + (size_t)(k0 + r) * ldkv + c4);
                if (all) vv = *reinterpret_cast<const float4*>(kb + (size_t)(k0 + r) * ldkv + GD + c4);
            }
            sm.Kt[c4 + 0][r] = kk.x; sm.Kt[c4 + 1][r] = kk.y; sm.Kt[c4 + 2][r] = kk.z; sm.Kt[c4 + 3][r] = kk.w;
            if (all) {
                sm.Vt[c4 + 0][r] = vv.x; sm.Vt[c4 + 1][r] = vv.y; sm.Vt[c4 + 2][r] = vv.z; sm.Vt[c4 + 3][r] = vv.w;
                *reinterpret_cast<float4*>(&sm.Kr[r][c4]) = kk;
            }
        }
        __syncthreads();
    };
    // s[i][j] = q_row . k_key (unscaled) -- and, with DP, p[i][j] = dO_row . v_key
    auto dots = [&](float (&s)[8][8], float (&p)[8][8], bool dp) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) { s[i][j] = 0.f; if (dp) p[i][j] = 0.f; }
#pragma unroll 2
        for (int d = 0; d < GD; ++d) {
            const float4 a0 = *reinterpret_cast<const float4*>(&sm.Qt[d][tq * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&sm.Qt[d][64 + tq * 4]);
            const float4 c0 = *reinterpret_cast<const float4*>(&sm.Kt[d][tk * 4]);
            const float4 c1 = *reinterpret_cast<const float4*>(&sm.Kt[d][32 + tk * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) s[i][j] = fmaf(av[i], cv[j], s[i][j]);
            if (dp) {
                const float4 g0 = *reinterpret_cast<const float4*>(&sm.Gt[d][tq * 4]);
                const float4 g1 = *reinterpret_cast<const float4*>(&sm.Gt[d][64 + tq * 4]);
                const float4 v0 = *reinterpret_cast<const float4*>(&sm.Vt[d][tk * 4]);
                const float4 v1 = *reinterpret_cast<const float4*>(&sm.Vt[d][32 + tk * 4]);
                const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                const float vv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) p[i][j] = fmaf(gv[i], vv[j], p[i][j]);
            }
        }
    };

    float m[8], l[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { m[i] = -INFINITY; l[i] = 0.f; }
    float s[8][8], p[8][8];
    // ---- pass 1: row max and sum of exp (as attention_maps_kernel)
    for (int k0 = 0; k0 < Nc; k0 += GK) {
        stage_keys(k0, false);
        dots(s, p, false);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = k0 + g_col(tk, j) < Nc ? s[i][j] * scale : -INFINITY;
            float mt = v[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) mt = fmaxf(mt, v[j]);
#pragma unroll
            for (int w = 4; w > 0; w >>= 1) mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, w));
            const float mnew = fmaxf(m[i], mt);
            float ps = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) ps += expf(v[j] - mnew);
#pragma unroll
            for (int w = 4; w > 0; w >>= 1) ps += __shfl_xor_sync(0xffffffffu, ps, w);
            l[i] = l[i] * expf(m[i] - mnew) + ps;
            m[i] = mnew;
        }
    }
    if (tk == 0) {      // the 8 threads of a row group hold the same values: kept in shared memory, out of pass 2's registers
#pragma unroll
        for (int i = 0; i < 8; ++i) { sm.Mr[g_row(tq, i)] = m[i]; sm.Lr[g_row(tq, i)] = 1.0f / l[i]; }
    }

    // ---- pass 2: W = P (dp - D) per key tile, dq += W k
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < Nc; k0 += GK) {
        stage_keys(k0, true);
        dots(s, p, true);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = g_row(tq, i);
            const float Di = sm.Dr[r], mi = sm.Mr[r], li = sm.Lr[r];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int key = g_col(tk, j);
                const float pr = k0 + key < Nc ? expf(s[i][j] * scale - mi) * li : 0.f;
                sm.Wt[key][g_row(tq, i)] = pr * (p[i][j] - Di);
            }
        }
        __syncthreads();
        const int kn = Nc - k0 < GK ? Nc - k0 : GK;
        for (int j = 0; j < kn; ++j) {
            const float4 w0 = *reinterpret_cast<const float4*>(&sm.Wt[j][tq * 4]);
            const float4 w1 = *reinterpret_cast<const float4*>(&sm.Wt[j][64 + tq * 4]);
            const float4 c0 = *reinterpret_cast<const float4*>(&sm.Kr[j][tk * 4]);
            const float4 c1 = *reinterpret_cast<const float4*>(&sm.Kr[j][32 + tk * 4]);
            const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
            const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[i][c] = fmaf(wv[i], cv[c], acc[i][c]);
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int r = r0 + g_row(tq, i);
        if (r >= N) continue;
        float* out = dq + (qb + r) * GD;
        *reinterpret_cast<float4*>(out + tk * 4) =
            make_float4(scale * acc[i][0], scale * acc[i][1], scale * acc[i][2], scale * acc[i][3]);
        *reinterpret_cast<float4*>(out + 32 + tk * 4) =
            make_float4(scale * acc[i][4], scale * acc[i][5], scale * acc[i][6], scale * acc[i][7]);
    }
}

unsigned grid1(long long n) { return (unsigned)((n + 255) / 256); }

}  // namespace

int fc_launch_act_fwd(const float* pre, int ldp, float* post, int ldq, long long M, int width, int act, int fast, cudaStream_t s) {
    FC_REQUIRE(pre && post && M > 0 && width > 0);
    act_fwd_kernel<<<grid1(M * width), 256, 0, s>>>(pre, ldp, post, ldq, M, width, act, fast);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

int fc_launch_act_bwd(float* d, int ldd, const float* pre, int ldp, long long M, int width, int act, cudaStream_t s) {
    FC_REQUIRE(d && pre && M > 0 && width > 0 && (act == FC_ACT_GELU || act == FC_ACT_RELU));
    act_bwd_kernel<<<grid1(M * width), 256, 0, s>>>(d, ldd, pre, ldp, M, width, act);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

int fc_launch_coupling_tail_bwd(const float* raw, int ldr, const float* x, int ldx, float* g, int ldg, int col0, int n2, float* dst,
                                int ldd, int M, cudaStream_t s) {
    FC_REQUIRE(raw && x && g && dst && M > 0 && n2 > 0);
    coupling_tail_bwd_kernel<<<grid1((long long)M * n2), 256, 0, s>>>(raw, ldr, x, ldx, g, ldg, col0, n2, dst, ldd, M);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

int fc_launch_augment_tail_bwd(const float* raw, int ldr, const float* eps, int S, const float* g, int ldg, int col0, float* dst,
                               int ldd, int M, cudaStream_t s) {
    FC_REQUIRE(raw && eps && g && dst && M > 0 && S > 0);
    augment_tail_bwd_kernel<<<grid1((long long)M * S), 256, 0, s>>>(raw, ldr, eps, S, g, ldg, col0, dst, ldd, M);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

int fc_launch_ln_bwd(const float* h, int ldh, const float* mu, const float* rstd, float* d, int ldd, int M, int width, cudaStream_t s) {
    FC_REQUIRE(h && mu && rstd && d && M > 0 && width > 0 && width <= 512);
    const int wpb = 8;
    ln_bwd_kernel<<<(M + wpb - 1) / wpb, wpb * 32, 0, s>>>(h, ldh, mu, rstd, d, ldd, M, width);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

int fc_launch_neg_copy(const float* z, int ldz, float* g, int ldg, long long M, int cols, cudaStream_t s) {
    FC_REQUIRE(z && g && M > 0 && cols > 0);
    neg_copy_kernel<<<grid1(M * cols), 256, 0, s>>>(z, ldz, g, ldg, M, cols);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

int fc_launch_attention_dq(const float* q, const float* kv, int ldkv, const float* o, const float* dO, float* dq, int B, int N,
                           int Nc, float scale, cudaStream_t stream) {
    FC_REQUIRE(q && kv && o && dO && dq && B > 0 && N > 0 && Nc > 0 && B <= 65535);
    FC_REQUIRE((ldkv & 3) == 0 && ldkv >= 2 * GD);
    FC_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(kv) | reinterpret_cast<uintptr_t>(dO) |
                 reinterpret_cast<uintptr_t>(dq)) & 15) == 0);
    int dev = 0;
    FC_CUDA_OK(cudaGetDevice(&dev));
    static std::atomic<uint64_t> configured{0};     // the dynamic shared-memory opt-in is per device
    if (!(configured.load(std::memory_order_acquire) & (1ull << (dev & 63)))) {
        FC_CUDA_OK(cudaFuncSetAttribute(attention_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DqSmem)));
        configured.fetch_or(1ull << (dev & 63), std::memory_order_release);
    }
    dim3 grid((N + GQ - 1) / GQ, B);
    const double pairs = (double)B * N * Nc;
    FcProfScope prof(FC_CLS_ATTENTION, 8.0 * GD * pairs, 4.0 * B * (4.0 * N * GD + 2.0 * Nc * 2 * GD), stream);
    attention_dq_kernel<<<grid, GTHREADS, sizeof(DqSmem), stream>>>(q, kv, ldkv, o, dO, dq, N, Nc, scale);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}
