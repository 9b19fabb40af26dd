// The cross-attention weights themselves, P = softmax(q k^T * scale) over the keys, reference models/perceiver.py:108-115
// (the `attn` tensor the reference's attention visualisation reads).  The flash kernels never form P, so this one writes it:
//
//   P[b, i, j] = exp(s_ij - m_i) / sum_j' exp(s_ij' - m_i),   s_ij = scale * (q[b*N + qidx[i], :] . k[b*Nc + j, :]),  m_i = max_j s_ij
//
// CTA = 128 query rows of one cloud, 128 threads, 8 x 8 scores per thread (rows tq*4.. and 64+tq*4.., keys tk*4.. and 32+tk*4..:
// every shared-memory read of a warp is one contiguous 128-byte wavefront).  Keys stream through shared memory in 64-key tiles
// twice: pass 1 keeps the online row max and sum, pass 2 recomputes s and writes the normalised weights (16-byte stores when
// Nc % 4 == 0; 8 lanes cover 128 contiguous bytes of a row).  The dot product is a sequential fp32 FMA chain over d = 0..63
// (packed FFMA2, two keys per instruction), so a weight depends on nothing but its own row and key: deterministic, independent
// of the batch, of the query list and of the other rows of the CTA.  Cost: 256 flop per weight against 4 bytes written.
#include <atomic>
#include "common.cuh"
#include "gemm.cuh"

namespace {

constexpr int MD = 64;        // head dim (single head, inner = 64)
constexpr int MQ = 128;       // query rows per CTA
constexpr int MK = 64;        // keys per tile
constexpr int MTHREADS = 128;
constexpr int MQLD = MQ + 4;  // padded leading dims of the transposed tiles
constexpr int MKLD = MK + 4;

struct MapsSmem {
    float Qt[MD][MQLD];   // Qt[d][row]
    float Kt[MD][MKLD];   // Kt[d][key]
};

// s[i][jp] = (score of row i, key 2jp) and (row i, key 2jp+1), unscaled; keys of pair jp: jp < 2 -> tk*4 + 2jp, else 32 + tk*4 + 2(jp-2)
__device__ __forceinline__ void score_tile(const MapsSmem& sm, int tq, int tk, float2 (&s)[8][4]) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int jp = 0; jp < 4; ++jp) s[i][jp] = make_float2(0.f, 0.f);
#pragma unroll 2
    for (int d = 0; d < MD; ++d) {
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
    }
}

__device__ __forceinline__ int key_of(int tk, int j) { return (j < 4 ? tk * 4 : 32 + tk * 4) + (j & 3); }

// VEC: 16-byte output stores (Nc % 4 == 0 and a 16-byte aligned output)
template <bool VEC>
__global__ void __launch_bounds__(MTHREADS, 3) attention_maps_kernel(const float* __restrict__ q, int ldq,
                                                                     const float* __restrict__ kv, int ldkv,
                                                                     const int32_t* __restrict__ qidx, int n_query,
                                                                     float* __restrict__ out, int N, int Nc, float scale) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MapsSmem& sm = *reinterpret_cast<MapsSmem*>(smem_raw);
    const int tid = threadIdx.x;
    const int tk = tid & 7;     // key group
    const int tq = tid >> 3;    // row group
    const int b = blockIdx.y;
    const int r0 = blockIdx.x * MQ;
    const float* qb = q + (size_t)b * N * ldq;
    const float* kb = kv + (size_t)b * Nc * ldkv;

    // Q rows of this CTA (picked through qidx), transposed; rows past n_query are zero and never stored
    for (int e = tid; e < MQ * (MD / 4); e += MTHREADS) {
        const int r = e / (MD / 4), c4 = (e % (MD / 4)) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r0 + r < n_query) {
            const int src = qidx ? qidx[r0 + r] : r0 + r;
            v = *reinterpret_cast<const float4*>(qb + (size_t)src * ldq + c4);
        }
        sm.Qt[c4 + 0][r] = v.x; sm.Qt[c4 + 1][r] = v.y; sm.Qt[c4 + 2][r] = v.z; sm.Qt[c4 + 3][r] = v.w;
    }
    auto stage_keys = [&](int k0) {
        __syncthreads();   // the previous tile is consumed (and, the first time, Q is staged)
        for (int e = tid; e < MK * (MD / 4); e += MTHREADS) {
            const int r = e / (MD / 4), c4 = (e % (MD / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k0 + r < Nc) v = *reinterpret_cast<const float4*>(kb + (size_t)(k0 + r) * ldkv + c4);
            sm.Kt[c4 + 0][r] = v.x; sm.Kt[c4 + 1][r] = v.y; sm.Kt[c4 + 2][r] = v.z; sm.Kt[c4 + 3][r] = v.w;
        }
        __syncthreads();
    };

    // ---- pass 1: row max and sum of exp, online over the key tiles.  fmaxf drops a NaN score, but its exp joins the sum,
    // so a NaN in q or k turns the whole row into NaN in pass 2 (never a silently renormalised row).
    float m[8], l[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { m[i] = -INFINITY; l[i] = 0.f; }
    float2 s[8][4];
    for (int k0 = 0; k0 < Nc; k0 += MK) {
        stage_keys(k0);
        score_tile(sm, tq, tk, s);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float raw = (j & 1) ? s[i][j >> 1].y : s[i][j >> 1].x;
                v[j] = k0 + key_of(tk, j) < Nc ? raw * scale : -INFINITY;
            }
            float mt = v[0];
#pragma unroll
            for (int j = 1; j < 8; ++j) mt = fmaxf(mt, v[j]);
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, o));
            const float mnew = fmaxf(m[i], mt);   // finite from the first tile on: it holds at least one key
            float ps = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) ps += expf(v[j] - mnew);
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) ps += __shfl_xor_sync(0xffffffffu, ps, o);
            l[i] = l[i] * expf(m[i] - mnew) + ps;
            m[i] = mnew;
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) l[i] = 1.0f / l[i];   // from here on: the reciprocal of the row sum

    // ---- pass 2: the same scores again, normalised and written
    for (int k0 = 0; k0 < Nc; k0 += MK) {
        stage_keys(k0);
        score_tile(sm, tq, tk, s);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int r = r0 + (i < 4 ? tq * 4 + i : 64 + tq * 4 + (i - 4));
            if (r >= n_query) continue;
            float* row = out + ((size_t)b * n_query + r) * (size_t)Nc;
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                const int key = k0 + (g == 0 ? tk * 4 : 32 + tk * 4);
                float p[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float raw = (e & 1) ? s[i][2 * g + (e >> 1)].y : s[i][2 * g + (e >> 1)].x;
                    p[e] = expf(raw * scale - m[i]) * l[i];
                }
                if (VEC && key + 3 < Nc) {
                    *reinterpret_cast<float4*>(row + key) = make_float4(p[0], p[1], p[2], p[3]);
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e) if (key + e < Nc) row[key + e] = p[e];
                }
            }
        }
    }
}

}  // namespace

int fc_launch_attention_maps(const float* q, int ldq, const float* kv, int ldkv, const int32_t* qidx, int n_query,
                             float* out, int B, int N, int Nc, float scale, cudaStream_t stream) {
    FC_REQUIRE(q && kv && out && B > 0 && N > 0 && Nc > 0 && n_query > 0);
    FC_REQUIRE(qidx || n_query == N);
    FC_REQUIRE((ldq & 3) == 0 && (ldkv & 3) == 0 && ldq >= MD && ldkv >= MD);
    FC_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(kv)) & 15) == 0);
    FC_REQUIRE(B <= 65535);
    int dev = 0;
    FC_CUDA_OK(cudaGetDevice(&dev));
    static std::atomic<uint64_t> configured{0};     // the dynamic shared-memory opt-in is per device
    if (!(configured.load(std::memory_order_acquire) & (1ull << (dev & 63)))) {
        FC_CUDA_OK(cudaFuncSetAttribute(attention_maps_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MapsSmem)));
        FC_CUDA_OK(cudaFuncSetAttribute(attention_maps_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MapsSmem)));
        configured.fetch_or(1ull << (dev & 63), std::memory_order_release);
    }
    const bool vec = (Nc & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    dim3 grid((n_query + MQ - 1) / MQ, B);
    const double elems = (double)B * n_query * Nc;
    FcProfScope prof(FC_CLS_ATTENTION, 4.0 * MD * elems, 4.0 * elems + 4.0 * B * ((double)n_query * MD + (double)Nc * MD), stream);
    if (vec) attention_maps_kernel<true><<<grid, MTHREADS, sizeof(MapsSmem), stream>>>(q, ldq, kv, ldkv, qidx, n_query, out, N, Nc, scale);
    else     attention_maps_kernel<false><<<grid, MTHREADS, sizeof(MapsSmem), stream>>>(q, ldq, kv, ldkv, qidx, n_query, out, N, Nc, scale);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}

extern "C" int fc_attention_maps(const float* q, int ldq, const float* kv, int ldkv, const int32_t* query_idx, int n_query,
                                 float* out, int B, int N, int Nc, float scale, fc_stream_t stream) {
    return fc_launch_attention_maps(q, ldq, kv, ldkv, query_idx, n_query, out, B, N, Nc, scale, (cudaStream_t)stream);
}
