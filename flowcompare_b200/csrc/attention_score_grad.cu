// The gradient of a point's log-likelihood with respect to its attention scores, reference models/perceiver.py:108-115 with
// sim = q k^T * scale, attn = sim.softmax(-1): what `sim.grad` holds after `sim.retain_grad()` and `log_prob.sum().backward()`.
// A point's log-prob depends on its own query row only, so with dO_i = d lp_i / d o_i from the input-gradient pass,
//
//   out[b, r, j] = d lp_i / d s_ij = P_ij (dO_i . v_j - D_i),   i = qidx[r],  D_i = dO_i . o_i,  P = softmax(s) over the keys
//
// the W of attention_dq_kernel (flow_grad.cu), which forms it tile by tile for dq and never writes it.  Laid out as
// attention_maps_kernel: CTA = 128 gathered query rows of one cloud, 128 threads, 8 x 8 values per thread (rows tq*4.. and
// 64+tq*4.., keys tk*4.. and 32+tk*4..).  Keys stream through shared memory in 64-key tiles twice: pass 1 keeps the online row
// max and sum, pass 2 recomputes s and dp = dO . v and writes W (16-byte stores when Nc % 4 == 0).  Every dot product is a
// sequential fp32 FMA chain over d = 0..63 (packed FFMA2, two keys per instruction), and P, D and W are formed exactly as in
// attention_dq_kernel, so a value depends on nothing but its own row and key: deterministic, independent of the batch and of
// the query list, and bitwise the W the dq kernel uses.  ACC adds each value to `out` with one rounded add (fc_flow_attention_
// score_grads sums blocks that way).  Cost: 384 flop per value against 4 bytes written (8 read-modify-written with ACC).
#include <atomic>
#include "common.cuh"
#include "gemm.cuh"

namespace {

constexpr int SD = 64;        // head dim (single head, inner = 64)
constexpr int SQ = 128;       // query rows per CTA
constexpr int SK = 64;        // keys per tile
constexpr int STHREADS = 128;
constexpr int SQLD = SQ + 4;  // padded leading dims of the transposed tiles
constexpr int SKLD = SK + 4;

struct ScoreGradSmem {
    float Qt[SD][SQLD];    // q transposed [d][row]
    float Gt[SD][SQLD];    // dO transposed
    float Kt[SD][SKLD];    // k transposed [d][key]
    float Vt[SD][SKLD];    // v transposed
    float Dr[SQ];          // D_i
    float Mr[SQ], Lr[SQ];  // row max of the scaled scores, 1 / row sum of exp (pass 1)
};

// s[i][jp] = q_row . k_key for keys 2jp, 2jp+1 of the thread's 8 (unscaled); with DP also p[i][jp] = dO_row . v_key
template <bool DP>
__device__ __forceinline__ void dots(const ScoreGradSmem& sm, int tq, int tk, float2 (&s)[8][4], float2 (&p)[8][4]) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int jp = 0; jp < 4; ++jp) { s[i][jp] = make_float2(0.f, 0.f); if (DP) p[i][jp] = make_float2(0.f, 0.f); }
#pragma unroll 2
    for (int d = 0; d < SD; ++d) {
        const float4 a0 = *reinterpret_cast<const float4*>(&sm.Qt[d][tq * 4]);
        const float4 a1 = *reinterpret_cast<const float4*>(&sm.Qt[d][64 + tq * 4]);
        const float4 c0 = *reinterpret_cast<const float4*>(&sm.Kt[d][tk * 4]);
        const float4 c1 = *reinterpret_cast<const float4*>(&sm.Kt[d][32 + tk * 4]);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float2 cv[4] = {make_float2(c0.x, c0.y), make_float2(c0.z, c0.w), make_float2(c1.x, c1.y), make_float2(c1.z, c1.w)};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int jp = 0; jp < 4; ++jp) s[i][jp] = __ffma2_rn(make_float2(av[i], av[i]), cv[jp], s[i][jp]);
        if (DP) {
            const float4 g0 = *reinterpret_cast<const float4*>(&sm.Gt[d][tq * 4]);
            const float4 g1 = *reinterpret_cast<const float4*>(&sm.Gt[d][64 + tq * 4]);
            const float4 v0 = *reinterpret_cast<const float4*>(&sm.Vt[d][tk * 4]);
            const float4 v1 = *reinterpret_cast<const float4*>(&sm.Vt[d][32 + tk * 4]);
            const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
            const float2 vv[4] = {make_float2(v0.x, v0.y), make_float2(v0.z, v0.w), make_float2(v1.x, v1.y), make_float2(v1.z, v1.w)};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int jp = 0; jp < 4; ++jp) p[i][jp] = __ffma2_rn(make_float2(gv[i], gv[i]), vv[jp], p[i][jp]);
        }
    }
}

__device__ __forceinline__ int sg_key(int tk, int j) { return (j < 4 ? tk * 4 : 32 + tk * 4) + (j & 3); }
__device__ __forceinline__ int sg_row(int tq, int i) { return i < 4 ? tq * 4 + i : 64 + tq * 4 + (i - 4); }
__device__ __forceinline__ float pick(const float2 (&t)[4], int j) { return (j & 1) ? t[j >> 1].y : t[j >> 1].x; }

// VEC: 16-byte output accesses (Nc % 4 == 0 and a 16-byte aligned output); ACC: out += value instead of out = value
template <bool VEC, bool ACC>
__global__ void __launch_bounds__(STHREADS, 2) attention_score_grad_kernel(const float* __restrict__ q, int ldq,
                                                                           const float* __restrict__ kv, int ldkv,
                                                                           const float* __restrict__ o, int ldo,
                                                                           const float* __restrict__ dO, int lddo,
                                                                           const int32_t* __restrict__ qidx, int n_query,
                                                                           float* __restrict__ out, int N, int Nc, float scale) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ScoreGradSmem& sm = *reinterpret_cast<ScoreGradSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int tk = tid & 7;     // key group
    const int tq = tid >> 3;    // row group
    const int b = blockIdx.y;
    const int r0 = blockIdx.x * SQ;
    const size_t rb = (size_t)b * N;
    const float* kb = kv + (size_t)b * Nc * ldkv;

    // q and dO rows of this CTA (picked through qidx), transposed; rows past n_query are zero and never stored
    for (int e = tid; e < SQ * (SD / 4); e += STHREADS) {
        const int r = e / (SD / 4), c4 = (e % (SD / 4)) * 4;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f), c = a;
        if (r0 + r < n_query) {
            const size_t src = rb + (qidx ? qidx[r0 + r] : r0 + r);
            a = *reinterpret_cast<const float4*>(q + src * ldq + c4);
            c = *reinterpret_cast<const float4*>(dO + src * lddo + c4);
        }
        sm.Qt[c4 + 0][r] = a.x; sm.Qt[c4 + 1][r] = a.y; sm.Qt[c4 + 2][r] = a.z; sm.Qt[c4 + 3][r] = a.w;
        sm.Gt[c4 + 0][r] = c.x; sm.Gt[c4 + 1][r] = c.y; sm.Gt[c4 + 2][r] = c.z; sm.Gt[c4 + 3][r] = c.w;
    }
    {   // D_i = dO_i . o_i, one row per thread (attention_dq_kernel's chain)
        float dd = 0.f;
        if (r0 + tid < n_query) {
            const size_t src = rb + (qidx ? qidx[r0 + tid] : r0 + tid);
            const float* op = o + src * ldo;
            const float* gp = dO + src * lddo;
            for (int d = 0; d < SD; ++d) dd = fmaf(gp[d], op[d], dd);
        }
        sm.Dr[tid] = dd;
    }
    auto stage_keys = [&](int k0, bool with_v) {
        __syncthreads();   // the previous tile is consumed (and, the first time, q / dO are staged)
        for (int e = tid; e < SK * (SD / 4); e += STHREADS) {
            const int r = e / (SD / 4), c4 = (e % (SD / 4)) * 4;
            float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
            if (k0 + r < Nc) {
                kk = *reinterpret_cast<const float4*>(kb + (size_t)(k0 + r) * ldkv + c4);
                if (with_v) vv = *reinterpret_cast<const float4*>(kb + (size_t)(k0 + r) * ldkv + SD + c4);
            }
            sm.Kt[c4 + 0][r] = kk.x; sm.Kt[c4 + 1][r] = kk.y; sm.Kt[c4 + 2][r] = kk.z; sm.Kt[c4 + 3][r] = kk.w;
            if (with_v) { sm.Vt[c4 + 0][r] = vv.x; sm.Vt[c4 + 1][r] = vv.y; sm.Vt[c4 + 2][r] = vv.z; sm.Vt[c4 + 3][r] = vv.w; }
        }
        __syncthreads();
    };

    // ---- pass 1: row max and sum of exp, online over the key tiles (as attention_maps_kernel: a NaN in q or k joins the sum
    // through its exp, so the whole row turns NaN in pass 2)
    float2 s[8][4], p[8][4];
    {
        float m[8], l[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { m[i] = -INFINITY; l[i] = 0.f; }
        for (int k0 = 0; k0 < Nc; k0 += SK) {
            stage_keys(k0, false);
            dots<false>(sm, tq, tk, s, p);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = k0 + sg_key(tk, j) < Nc ? pick(s[i], j) * scale : -INFINITY;
                float mt = v[0];
#pragma unroll
                for (int j = 1; j < 8; ++j) mt = fmaxf(mt, v[j]);
#pragma unroll
                for (int w = 4; w > 0; w >>= 1) mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, w));
                const float mnew = fmaxf(m[i], mt);   // finite from the first tile on: it holds at least one key
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
            for (int i = 0; i < 8; ++i) { sm.Mr[sg_row(tq, i)] = m[i]; sm.Lr[sg_row(tq, i)] = 1.0f / l[i]; }
        }
    }

    // ---- pass 2: the scores again and dp; W = P (dp - D) written (the first stage_keys orders Mr / Lr before their reads)
    for (int k0 = 0; k0 < Nc; k0 += SK) {
        stage_keys(k0, true);
        dots<true>(sm, tq, tk, s, p);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int rl = sg_row(tq, i);
            const int r = r0 + rl;
            if (r >= n_query) continue;
            const float Di = sm.Dr[rl], mi = sm.Mr[rl], li = sm.Lr[rl];
            float* row = out + ((size_t)b * n_query + r) * (size_t)Nc;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                const int key = k0 + (g == 0 ? tk * 4 : 32 + tk * 4);
                float w[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float pr = expf(pick(s[i], 4 * g + e) * scale - mi) * li;
                    w[e] = pr * (pick(p[i], 4 * g + e) - Di);
                }
                if (VEC && key + 3 < Nc) {
                    float4* dst = reinterpret_cast<float4*>(row + key);
                    if (ACC) {
                        const float4 a = *dst;
                        *dst = make_float4(__fadd_rn(a.x, w[0]), __fadd_rn(a.y, w[1]), __fadd_rn(a.z, w[2]), __fadd_rn(a.w, w[3]));
                    } else {
                        *dst = make_float4(w[0], w[1], w[2], w[3]);
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (key + e < Nc) row[key + e] = ACC ? __fadd_rn(row[key + e], w[e]) : w[e];
                }
            }
        }
    }
}

template <bool VEC, bool ACC>
void launch(dim3 grid, cudaStream_t stream, const float* q, int ldq, const float* kv, int ldkv, const float* o, int ldo,
            const float* dO, int lddo, const int32_t* qidx, int n_query, float* out, int N, int Nc, float scale) {
    attention_score_grad_kernel<VEC, ACC><<<grid, STHREADS, sizeof(ScoreGradSmem), stream>>>(q, ldq, kv, ldkv, o, ldo, dO, lddo, qidx,
                                                                                            n_query, out, N, Nc, scale);
}

}  // namespace

int fc_launch_attention_score_grad(const float* q, int ldq, const float* kv, int ldkv, const float* o, int ldo, const float* dO,
                                   int lddo, const int32_t* qidx, int n_query, float* out, int accumulate, int B, int N, int Nc,
                                   float scale, cudaStream_t stream) {
    FC_REQUIRE(q && kv && o && dO && out && B > 0 && N > 0 && Nc > 0 && n_query > 0);
    FC_REQUIRE(qidx || n_query == N);
    FC_REQUIRE((ldq & 3) == 0 && (ldkv & 3) == 0 && (lddo & 3) == 0 && ldq >= SD && ldkv >= 2 * SD && ldo >= SD && lddo >= SD);
    FC_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(kv) | reinterpret_cast<uintptr_t>(dO)) & 15) == 0);
    FC_REQUIRE(B <= 65535);
    int dev = 0;
    FC_CUDA_OK(cudaGetDevice(&dev));
    static std::atomic<uint64_t> configured{0};     // the dynamic shared-memory opt-in is per device
    if (!(configured.load(std::memory_order_acquire) & (1ull << (dev & 63)))) {
        const int bytes = (int)sizeof(ScoreGradSmem);
        FC_CUDA_OK(cudaFuncSetAttribute(attention_score_grad_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        FC_CUDA_OK(cudaFuncSetAttribute(attention_score_grad_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        FC_CUDA_OK(cudaFuncSetAttribute(attention_score_grad_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        FC_CUDA_OK(cudaFuncSetAttribute(attention_score_grad_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        configured.fetch_or(1ull << (dev & 63), std::memory_order_release);
    }
    const bool vec = (Nc & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    dim3 grid((n_query + SQ - 1) / SQ, B);
    const double elems = (double)B * n_query * Nc;
    FcProfScope prof(FC_CLS_ATTENTION, 6.0 * SD * elems,
                     (accumulate ? 8.0 : 4.0) * elems + 4.0 * B * ((double)n_query * 3 * SD + (double)Nc * 2 * SD), stream);
    if (vec) {
        if (accumulate) launch<true, true>(grid, stream, q, ldq, kv, ldkv, o, ldo, dO, lddo, qidx, n_query, out, N, Nc, scale);
        else            launch<true, false>(grid, stream, q, ldq, kv, ldkv, o, ldo, dO, lddo, qidx, n_query, out, N, Nc, scale);
    } else {
        if (accumulate) launch<false, true>(grid, stream, q, ldq, kv, ldkv, o, ldo, dO, lddo, qidx, n_query, out, N, Nc, scale);
        else            launch<false, false>(grid, stream, q, ldq, kv, ldkv, o, ldo, dO, lddo, qidx, n_query, out, N, Nc, scale);
    }
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

extern "C" int fc_attention_score_grad(const float* q, int ldq, const float* kv, int ldkv, const float* o, int ldo, const float* dO,
                                       int lddo, const int32_t* query_idx, int n_query, float* out, int accumulate, int B, int N,
                                       int Nc, float scale, fc_stream_t stream) {
    return fc_launch_attention_score_grad(q, ldq, kv, ldkv, o, ldo, dO, lddo, query_idx, n_query, out, accumulate, B, N, Nc, scale,
                                          (cudaStream_t)stream);
}
