// PAConv context embedder: `PointNet2SSGSeg.forward` (reference
// models/scene_seg_PAConv/model/pointnet2/pointnet2_paconv_seg.py:63-82) =
//   4 x SA  (_PointNet2SAModuleBase.forward, pointnet2_paconv_modules.py:20-61): furthest point sampling,
//           kNN grouping (QueryAndGroup, lib/pointops/functions/pointops.py:557-594), 3 PAConv layers
//           (paconv.py:107-153: ScoreNet :31-54 softmax scores over m=8 weight-bank kernels, assign_score
//           paconv_util.py:52-56, BN, ReLU), max over the K=32 neighbours
//   4 x FP  (PointNet2FPModule.forward :206-238): 3-NN inverse-distance interpolation + SharedMLP
//   out MLP (models/nets.py:19-30)
//
// Layout: everything point-major / edge-major ([points, C] and [edges, C] with edge = (cloud, centre, k)).
// The weight-bank product + score-weighted sum of one PAConv layer,
//     out[e, o] = sum_m s_m(e) * sum_c x[e, c] * WB[c, m*Cout + o],
// is evaluated as ONE GEMM over the expanded input X'[e, (m, c)] = s_m(e) * x[e, c] (the reference's own
// fused form, lib/paconv_lib/src/gpu/assign_score_withk_gpu.cu:18-49, restated as a matrix product), so BN
// and ReLU ride in the GEMM epilogue and the [edges, m, Cout] intermediate of the reference never exists.
// The index-producing kernels (FPS, heap kNN, 3-NN) restate the reference algorithms including their tie
// behaviour and are checked bit-for-bit against oracle/pointops_ref.c.
#include "model.cuh"
#include <new>

namespace {

constexpr int PA_M = 8;          // weight-bank kernels
constexpr int PA_SH = 16;        // ScoreNet hidden width
constexpr int PA_K = 32;         // neighbours per centre
constexpr int PA_SCORE_FLOATS = PA_SH * 3 + PA_SH + PA_M * PA_SH + PA_M;   // w0[16][3], b0[16], w1[8][16], b1[8]

struct PaLayer { const float* score; FcLinear lin; int Cin, Cout; };
struct PaSA { PaLayer layer[3]; int npoint; int Cin0; };     // Cin0 = 3 + feature channels entering the level
struct PaFP { FcLinear lin[3]; int n_layers; int Cin; };
struct PaModel {
    PaSA sa[4];
    PaFP fp[4];
    int c_feat;       // input feature channels (input_dim - 3)
};

// the contraction nvcc applies to the reference's `dx*dx + dy*dy + dz*dz` (read off the SASS of its kernels: FMUL dy*dy, FFMA dx, FFMA dz)
__device__ __forceinline__ float sqdist3(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = ax - bx, dy = ay - by, dz = az - bz;
    return fmaf(dz, dz, fmaf(dx, dx, dy * dy));
}

// pts [B,N,d_in] -> xyz [B,N,3], feat [B,N,ldf] (first c columns)
__global__ void split_points_kernel(const float* __restrict__ pts, int d_in, long long total, float* __restrict__ xyz,
                                    float* __restrict__ feat, int ldf) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float* p = pts + i * d_in;
    xyz[i * 3 + 0] = p[0]; xyz[i * 3 + 1] = p[1]; xyz[i * 3 + 2] = p[2];
    for (int c = 3; c < d_in; ++c) feat[i * ldf + c - 3] = p[c];
}

// K2, furthest point sampling.  The algorithm is sequential in the number of samples (each pick depends on the last), so
// the kernel is latency bound: what matters is the length of ONE iteration.  One CTA per cloud; every thread keeps its
// points AND their running minimum distances in registers (PT points per thread), the cloud's coordinates sit in shared
// memory for the broadcast read of the last pick, and the block arg-max is two warp-shuffle reductions around ONE barrier
// (double-buffered partials) -- the reference design (lib/pointops/src/sampling/sampling_cuda_kernel.cu:58-168) re-reads
// xyz and `temp` from global memory every iteration and walks a 10-level shared-memory tree with a barrier per level.
// Tie rule (needed for bit-exact indices on clouds with duplicate points; checked against the reference's compiled
// kernel, tests/test_pointops_gpu.py): the reference scans point k in thread k % block of ITS launch (block = 2^floor(log2 n)
// <= 1024 threads; first maximum within a thread) and then walks a halving tree in which slot s meets slot s + h and the
// LOWER slot keeps ties.  Two equal candidates therefore meet at the lowest bit in which their thread ids differ and the
// one with a 0 there wins: the order is the BIT-REVERSED thread id, then the index within the thread.  That key is carried
// through the reduction, so the result does not depend on this kernel's own block size.  log2bs < 0: lowest index wins.
template <int PT>
__global__ void __launch_bounds__(1024) fps_kernel(const float* __restrict__ xyz, int n, int m, int log2bs,
                                                   int32_t* __restrict__ idx, float* __restrict__ new_xyz, int xyz_in_smem) {
    extern __shared__ float fps_sm[];
    __shared__ unsigned long long part[2][32];
    const int b = blockIdx.x, tid = threadIdx.x, bs = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = bs >> 5;
    const float* x = xyz + (size_t)b * n * 3;
    float px[PT], py[PT], pz[PT], dist[PT];
    unsigned prio[PT];
    const unsigned bs_ref = log2bs >= 0 ? 1u << log2bs : 0u;
    const unsigned R = log2bs >= 0 ? ((unsigned)n + bs_ref - 1) >> log2bs : 1u;   // points per reference thread
#pragma unroll
    for (int i = 0; i < PT; ++i) {
        const int k = tid + i * bs;
        px[i] = py[i] = pz[i] = 0.f; dist[i] = 1e10f; prio[i] = 0xffffffffu;
        if (k < n) {
            px[i] = x[k * 3 + 0]; py[i] = x[k * 3 + 1]; pz[i] = x[k * 3 + 2];
            prio[i] = log2bs > 0 ? (__brev((unsigned)k & (bs_ref - 1)) >> (32 - log2bs)) * R + ((unsigned)k >> log2bs) : (unsigned)k;
            if (xyz_in_smem) { fps_sm[k * 3 + 0] = px[i]; fps_sm[k * 3 + 1] = py[i]; fps_sm[k * 3 + 2] = pz[i]; }
        }
    }
    const float* xs = xyz_in_smem ? fps_sm : x;
    if (tid == 0) {
        idx[(size_t)b * m] = 0;
        if (new_xyz) { float* o = new_xyz + (size_t)b * m * 3; o[0] = x[0]; o[1] = x[1]; o[2] = x[2]; }
    }
    __syncthreads();
    int old = 0;
    for (int j = 1; j < m; ++j) {
        const float ox = xs[old * 3 + 0], oy = xs[old * 3 + 1], oz = xs[old * 3 + 2];
        // key = (distance bits, ~priority): distances are >= 0, so their bit patterns order like the values
        unsigned long long best = 0ull;
#pragma unroll
        for (int i = 0; i < PT; ++i) {
            const float d2 = fminf(sqdist3(px[i], py[i], pz[i], ox, oy, oz), dist[i]);
            dist[i] = d2;
            const unsigned long long key = ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)(~prio[i]);
            if (prio[i] != 0xffffffffu && key > best) best = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffffu, best, o); best = v > best ? v : best; }
        if (lane == 0) part[j & 1][warp] = best;
        __syncthreads();
        best = lane < nwarps ? part[j & 1][lane] : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(0xffffffffu, best, o); best = v > best ? v : best; }
        const unsigned pr = ~(unsigned)best;
        old = log2bs > 0 ? (int)(((pr % R) << log2bs) + (__brev(pr / R) >> (32 - log2bs))) : (int)pr;
        if (tid == 0) {
            idx[(size_t)b * m + j] = old;
            if (new_xyz) { float* o = new_xyz + ((size_t)b * m + j) * 3; o[0] = xs[old * 3 + 0]; o[1] = xs[old * 3 + 1]; o[2] = xs[old * 3 + 2]; }
        }
    }
}

// K1, k-nearest-neighbour query: one thread per query, the reference's max-heap algorithm step for step (strict < replaces
// the root, heap-sort at the end; slots never filled when k > n keep index 0) because the ORDER of equal-distance
// neighbours in its output is an artefact of that heap and neighbour 0 is PAConv's centre (paconv.py:123).  What changes is
// where things live: the reference keeps the heap in per-thread LOCAL memory (dynamically indexed best_dist[100] /
// best_idx[100], lib/pointops/src/knnquery_heap/knnquery_heap_cuda_kernel.cu:67-68) and every thread streams the whole
// cloud from global memory; here the heaps of a CTA's queries live in shared memory ([slot][query], padded: conflict free
// for the sift and for the coalesced write-out) and the candidates are staged once per CTA in shared-memory tiles.
constexpr int KH_Q = 128;      // queries per CTA
constexpr int KH_T = 512;      // candidates per tile
__device__ __forceinline__ void heap_sift(float* d, int* ix, int size) {   // d / ix: this query's column, stride KH_Q + 1
    constexpr int S = KH_Q + 1;
    int root = 0;
    for (;;) {
        int child = 2 * root + 1;
        if (child >= size) return;
        if (child + 1 < size && d[(child + 1) * S] > d[child * S]) ++child;
        const float dr = d[root * S], dc = d[child * S];
        if (dr > dc) return;
        d[root * S] = dc; d[child * S] = dr;
        const int ti = ix[root * S]; ix[root * S] = ix[child * S]; ix[child * S] = ti;
        root = child;
    }
}
__global__ void __launch_bounds__(KH_Q) knn_heap_kernel(const float* __restrict__ xyz, const float* __restrict__ queries, int n, int m,
                                                         int k, int32_t* __restrict__ idx, float* __restrict__ dist2) {
    extern __shared__ float kh_sm[];
    constexpr int S = KH_Q + 1;
    float* hd = kh_sm;                                      // [k][S]
    int* hi = reinterpret_cast<int*>(kh_sm + (size_t)k * S);   // [k][S]
    float* tile = kh_sm + (size_t)2 * k * S;                // [KH_T][3]
    const int b = blockIdx.y, tid = threadIdx.x;
    const int q = blockIdx.x * KH_Q + tid;
    const float* x = xyz + (size_t)b * n * 3;
    float cx = 0.f, cy = 0.f, cz = 0.f;
    if (q < m) { const float* c = queries + ((size_t)b * m + q) * 3; cx = c[0]; cy = c[1]; cz = c[2]; }
    float* d = hd + tid; int* ix = hi + tid;
    for (int i = 0; i < k; ++i) { d[i * S] = 1e10f; ix[i * S] = 0; }
    for (int t0 = 0; t0 < n; t0 += KH_T) {
        const int cnt = min(KH_T, n - t0);
        __syncthreads();
        for (int e = tid; e < cnt * 3; e += KH_Q) tile[e] = x[(size_t)t0 * 3 + e];
        __syncthreads();
        if (q < m) {
            float root = d[0];
            for (int i = 0; i < cnt; ++i) {
                const float d2 = sqdist3(cx, cy, cz, tile[i * 3 + 0], tile[i * 3 + 1], tile[i * 3 + 2]);
                if (d2 < root) { d[0] = d2; ix[0] = t0 + i; heap_sift(d, ix, k); root = d[0]; }
            }
        }
    }
    if (q < m)
        for (int i = k - 1; i > 0; --i) {
            const float td = d[0]; d[0] = d[i * S]; d[i * S] = td;
            const int ti = ix[0]; ix[0] = ix[i * S]; ix[i * S] = ti;
            heap_sift(d, ix, i);
        }
    __syncthreads();
    // coalesced write-out: consecutive threads write consecutive slots of one query
    const int q0 = blockIdx.x * KH_Q;
    for (int e = tid; e < KH_Q * k; e += KH_Q) {
        const int ql = e / k, sl = e % k;
        if (q0 + ql < m) {
            const size_t o = ((size_t)b * m + q0 + ql) * k + sl;
            idx[o] = hi[sl * S + ql];
            if (dist2) dist2[o] = hd[sl * S + ql];
        }
    }
}

// QueryAndGroup: edge e = (b, centre j, k).  f0[e] = [xyz[idx] - new_xyz[j] | feat[idx]]  (width 3 + C),
// dxyz[e] = xyz[idx[e]] - xyz[idx[b,j,0]]  (PAConv's "centre" is neighbour 0, paconv.py:123)
__global__ void group_kernel(const float* __restrict__ xyz, const float* __restrict__ feat, int ldfeat, int C,
                             const float* __restrict__ new_xyz, const int32_t* __restrict__ idx, int n, int m,
                             long long edges, float* __restrict__ f0, int ldf0, float* __restrict__ dxyz) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= edges) return;
    const long long grp = e / PA_K;            // (b*m + j)
    const long long b = grp / m;
    const int src = idx[e], src0 = idx[grp * PA_K];
    const float* px = xyz + ((size_t)b * n + src) * 3;
    const float* p0 = xyz + ((size_t)b * n + src0) * 3;
    const float* cx = new_xyz + (size_t)grp * 3;
    float* o = f0 + (size_t)e * ldf0;
    o[0] = px[0] - cx[0]; o[1] = px[1] - cx[1]; o[2] = px[2] - cx[2];
    const float* pf = feat + ((size_t)b * n + src) * ldfeat;
    for (int c = 0; c < C; ++c) o[3 + c] = pf[c];
    dxyz[e * 3 + 0] = px[0] - p0[0]; dxyz[e * 3 + 1] = px[1] - p0[1]; dxyz[e * 3 + 2] = px[2] - p0[2];
}

// One CTA per centre (32 edges).  ScoreNet (conv 3->16 with BN folded, ReLU, conv 16->8 + bias, softmax over the 8
// kernels) then X'[e, m*2C + c] = s_m(e) * x[e, c],  x = [f - f(k=0) | f]   (kernel_input='neighbor', paconv.py:125-128)
__global__ void __launch_bounds__(256) paconv_expand_kernel(const float* __restrict__ f, int ldf, int C,
                                                            const float* __restrict__ dxyz, const float* __restrict__ score,
                                                            float* __restrict__ X, int ldx) {
    __shared__ float s[PA_K][PA_M];
    __shared__ float sp[PA_SCORE_FLOATS];
    const long long e0 = (long long)blockIdx.x * PA_K;
    for (int i = threadIdx.x; i < PA_SCORE_FLOATS; i += blockDim.x) sp[i] = score[i];
    __syncthreads();
    if (threadIdx.x < PA_K) {
        const float* w0 = sp; const float* b0 = sp + PA_SH * 3; const float* w1 = b0 + PA_SH; const float* b1 = w1 + PA_M * PA_SH;
        const float* d = dxyz + (e0 + threadIdx.x) * 3;
        float h[PA_SH];
#pragma unroll
        for (int i = 0; i < PA_SH; ++i) {
            const float v = fmaf(w0[i * 3 + 2], d[2], fmaf(w0[i * 3 + 1], d[1], w0[i * 3 + 0] * d[0])) + b0[i];
            h[i] = v > 0.f ? v : 0.f;
        }
        float z[PA_M], mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < PA_M; ++k) {
            float acc = b1[k];
#pragma unroll
            for (int i = 0; i < PA_SH; ++i) acc = fmaf(w1[k * PA_SH + i], h[i], acc);
            z[k] = acc; mx = fmaxf(mx, acc);
        }
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < PA_M; ++k) { z[k] = expf(z[k] - mx); sum += z[k]; }
#pragma unroll
        for (int k = 0; k < PA_M; ++k) s[threadIdx.x][k] = z[k] / sum;
    }
    __syncthreads();
    const int C2 = 2 * C;
    const float* fc = f + (size_t)e0 * ldf;               // centre row (k = 0)
    for (int i = threadIdx.x; i < PA_K * C2; i += blockDim.x) {
        const int k = i / C2, c = i % C2;
        const float* fr = f + (size_t)(e0 + k) * ldf;
        const float v = c < C ? fr[c] - fc[c] : fr[c - C];
        float* o = X + (size_t)(e0 + k) * ldx + c;
#pragma unroll
        for (int mm = 0; mm < PA_M; ++mm) o[mm * C2] = s[k][mm] * v;
    }
}

// max over the K neighbours: [groups*K, C] -> [groups, C]
__global__ void max_over_k_kernel(const float* __restrict__ f, int ldf, int C, long long groups, float* __restrict__ out, int ldo) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= groups * C) return;
    const long long g = i / C; const int c = (int)(i % C);
    const float* p = f + (size_t)g * PA_K * ldf + c;
    float m = p[0];
#pragma unroll 4
    for (int k = 1; k < PA_K; ++k) m = fmaxf(m, p[(size_t)k * ldf]);
    out[(size_t)g * ldo + c] = m;
}

// K5 + FP weights: one thread per unknown point; strict < insertion (lower index wins ties); the known points are staged once
// per CTA in shared memory (the reference re-reads them from global memory in every thread,
// lib/pointops/src/interpolation/interpolation_cuda_kernel.cu:134-176).  Outputs: idx, and either the reference's squared
// distances (op-level entry point) or the FP module's weights w = (1/(sqrt(d2)+1e-8)) / sum (pointnet2_paconv_modules.py:225-228).
constexpr int NN_T = 1024;
__global__ void __launch_bounds__(128) three_nn_kernel(const float* __restrict__ unknown, const float* __restrict__ known, int n, int m,
                                                       int32_t* __restrict__ idx, float* __restrict__ w, float* __restrict__ dist2) {
    __shared__ float tile[NN_T * 3];
    const int b = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const float* kx = known + (size_t)b * m * 3;
    float ux = 0.f, uy = 0.f, uz = 0.f;
    if (p < n) { const float* u = unknown + ((size_t)b * n + p) * 3; ux = u[0]; uy = u[1]; uz = u[2]; }
    double b1 = 1e40, b2 = 1e40, b3 = 1e40;
    int i1 = 0, i2 = 0, i3 = 0;
    for (int t0 = 0; t0 < m; t0 += NN_T) {
        const int cnt = min(NN_T, m - t0);
        __syncthreads();
        for (int e = threadIdx.x; e < cnt * 3; e += blockDim.x) tile[e] = kx[(size_t)t0 * 3 + e];
        __syncthreads();
        for (int k = 0; k < cnt; ++k) {
            const float d = sqdist3(ux, uy, uz, tile[k * 3 + 0], tile[k * 3 + 1], tile[k * 3 + 2]);
            if (d < b1) { b3 = b2; i3 = i2; b2 = b1; i2 = i1; b1 = d; i1 = t0 + k; }
            else if (d < b2) { b3 = b2; i3 = i2; b2 = d; i2 = t0 + k; }
            else if (d < b3) { b3 = d; i3 = t0 + k; }
        }
    }
    if (p >= n) return;
    const size_t o = ((size_t)b * n + p) * 3;
    idx[o + 0] = i1; idx[o + 1] = i2; idx[o + 2] = i3;
    if (dist2) { dist2[o + 0] = (float)b1; dist2[o + 1] = (float)b2; dist2[o + 2] = (float)b3; }
    if (w) {
        const float r1 = 1.0f / (sqrtf((float)b1) + 1e-8f), r2 = 1.0f / (sqrtf((float)b2) + 1e-8f), r3 = 1.0f / (sqrtf((float)b3) + 1e-8f);
        const float norm = (r1 + r2) + r3;
        w[o + 0] = r1 / norm; w[o + 1] = r2 / norm; w[o + 2] = r3 / norm;
    }
}
__global__ void interp_concat_kernel(const float* __restrict__ known_feat, int ldk, int C2, const float* __restrict__ unk_feat,
                                     int ldu, int C1, const int32_t* __restrict__ idx, const float* __restrict__ w, int n, int m,
                                     long long total_pts, float* __restrict__ out, int ldo) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int Ct = C2 + C1;
    if (i >= total_pts * Ct) return;
    const long long p = i / Ct; const int c = (int)(i % Ct);
    float v;
    if (c < C2) {
        const long long b = p / n;
        const float* kf = known_feat + (size_t)b * m * ldk + c;
        const int32_t* ix = idx + p * 3; const float* ww = w + p * 3;
        // the contraction nvcc applies to the reference's `w0*p0 + w1*p1 + w2*p2` (interpolation_cuda_kernel.cu:194): the first product is
        // fused into the second's rounded value, then the third is fused on top
        v = fmaf(ww[2], kf[(size_t)ix[2] * ldk], fmaf(ww[0], kf[(size_t)ix[0] * ldk], ww[1] * kf[(size_t)ix[1] * ldk]));
    } else {
        v = unk_feat[(size_t)p * ldu + (c - C2)];
    }
    out[(size_t)p * ldo + c] = v;
}

int fps_threads(int n) {   // block size of the REFERENCE launcher (opt_n_threads, cuda_utils.h:15-18): fixes its tie order
    const int p = (int)(log((double)n) / log(2.0));
    int t = 1 << p;
    if (t > 1024) t = 1024;
    if (t < 1) t = 1;
    return t;
}

// tie_block: 0 = the reference launcher's rule (2^floor(log2 n) <= 1024), > 0 explicit, < 0 lowest index wins
int launch_fps(const float* xyz, int B, int n, int m, int tie_block, int32_t* idx, float* new_xyz, cudaStream_t s) {
    FC_REQUIRE(xyz && idx && B > 0 && n > 0 && m > 0 && m <= n && n <= 32768 && B <= 65535);
    const int bs_ref = tie_block == 0 ? fps_threads(n) : tie_block;
    FC_REQUIRE(tie_block < 0 || (bs_ref & (bs_ref - 1)) == 0);     // the reference's blocks are powers of two
    int log2bs = -1;
    if (tie_block >= 0) { log2bs = 0; while ((1 << log2bs) < bs_ref) ++log2bs; }
    int threads = fc_round_up(n, 32);
    if (threads > 1024) threads = 1024;
    const int pt = (n + threads - 1) / threads;
    const int in_smem = (size_t)n * 12 <= 40 * 1024;
    const size_t smem = in_smem ? (size_t)n * 12 : 0;
#define FC_FPS_CASE(P) fps_kernel<P><<<B, threads, smem, s>>>(xyz, n, m, log2bs, idx, new_xyz, in_smem)
    if (pt <= 1) FC_FPS_CASE(1); else if (pt <= 2) FC_FPS_CASE(2); else if (pt <= 4) FC_FPS_CASE(4);
    else if (pt <= 8) FC_FPS_CASE(8); else if (pt <= 16) FC_FPS_CASE(16); else FC_FPS_CASE(32);
#undef FC_FPS_CASE
    fc_count_launch(); FC_LAUNCH_OK();
    return FC_OK;
}

int launch_knn_heap(const float* xyz, const float* queries, int B, int n, int m, int k, int32_t* idx, float* dist2, cudaStream_t s) {
    FC_REQUIRE(xyz && queries && idx && B > 0 && n > 0 && m > 0 && k >= 1 && k <= 40 && B <= 65535);
    const size_t smem = ((size_t)2 * k * (KH_Q + 1) + KH_T * 3) * 4;   // <= 47.4 KB at k = 40
    knn_heap_kernel<<<dim3((m + KH_Q - 1) / KH_Q, B), KH_Q, smem, s>>>(xyz, queries, n, m, k, idx, dist2);
    fc_count_launch(); FC_LAUNCH_OK();
    return FC_OK;
}

int launch_three_nn(const float* unknown, const float* known, int B, int n, int m, int32_t* idx, float* w, float* dist2, cudaStream_t s) {
    FC_REQUIRE(unknown && known && idx && B > 0 && n > 0 && m > 0 && B <= 65535);
    three_nn_kernel<<<dim3((n + 127) / 128, B), 128, 0, s>>>(unknown, known, n, m, idx, w, dist2);
    fc_count_launch(); FC_LAUNCH_OK();
    return FC_OK;
}

// K4 (grouping) in point-major layout: out[b, j, kk, :] = feat[b, idx[b, j, kk], :]
__global__ void gather_rows_kernel(const float* __restrict__ feat, int ldf, int C, const int32_t* __restrict__ idx, int n, long long rows_per_cloud,
                                   long long total, float* __restrict__ out, int ldo) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total * C) return;
    const long long r = i / C; const int c = (int)(i % C);
    const long long b = r / rows_per_cloud;
    out[(size_t)r * ldo + c] = feat[((size_t)b * n + idx[r]) * ldf + c];
}

const int SA_W[4][4] = {{0, 32, 32, 64}, {64, 64, 64, 128}, {128, 128, 128, 256}, {256, 256, 256, 512}};   // [i][0] + 3 (+c for i=0)
const int FP_N[4] = {3, 2, 2, 2};
const int FP_W[4][4] = {{128, 128, 128, 128}, {320, 256, 128, 0}, {384, 256, 256, 0}, {768, 256, 256, 0}};  // [0][0] + c

struct PaWs {
    float *xyz[5], *feat[5], *dxyz, *fA, *fB, *X, *fpcat, *fph, *w3, *hA, *hB;
    int32_t *fidx, *kidx, *idx3;
    int n[5], ldfeat[5];
    int64_t total;
};

PaWs carve_pa(const fc_embedder* e, const PaModel* pm, int B, int Nc, void* base) {
    PaWs w{};
    int64_t off = 0;
    auto take = [&](int64_t bytes) { char* p = base ? reinterpret_cast<char*>(base) + off : nullptr; off += fc_round_up_ll(bytes, 256); return p; };
    const int cfeat[5] = {pm->c_feat, 64, 128, 256, 512};
    w.n[0] = Nc;
    for (int i = 0; i < 4; ++i) w.n[i + 1] = pm->sa[i].npoint;
    for (int i = 0; i < 5; ++i) {
        w.ldfeat[i] = fc_round_up(cfeat[i], 4);
        w.xyz[i] = (float*)take((int64_t)B * w.n[i] * 3 * 4);
        w.feat[i] = (float*)take((int64_t)B * w.n[i] * w.ldfeat[i] * 4);
    }
    int64_t max_edges = 0, max_f = 0, max_x = 0;
    for (int i = 0; i < 4; ++i) {
        const int64_t edges = (int64_t)B * w.n[i + 1] * PA_K;
        max_edges = edges > max_edges ? edges : max_edges;
        for (int j = 0; j < 3; ++j) {
            const int cin = pm->sa[i].layer[j].Cin, cout = pm->sa[i].layer[j].Cout;
            const int64_t fin = edges * fc_round_up(cin, 4), fout = edges * cout, xx = edges * (int64_t)PA_M * 2 * cin;
            max_f = fin > max_f ? fin : max_f; max_f = fout > max_f ? fout : max_f; max_x = xx > max_x ? xx : max_x;
        }
    }
    w.fidx = (int32_t*)take((int64_t)B * w.n[1] * 4);
    w.kidx = (int32_t*)take(max_edges * 4);
    w.dxyz = (float*)take(max_edges * 3 * 4);
    w.fA = (float*)take(max_f * 4);
    w.fB = (float*)take(max_f * 4);
    w.X = (float*)take(max_x * 4);
    w.idx3 = (int32_t*)take((int64_t)B * Nc * 3 * 4);
    w.w3 = (float*)take((int64_t)B * Nc * 3 * 4);
    w.fpcat = (float*)take((int64_t)B * Nc * 768 * 4 / 1 > 0 ? (int64_t)B * Nc * 132 * 4 + (int64_t)B * w.n[1] * 768 * 4 : 0);
    w.fph = (float*)take((int64_t)B * Nc * 256 * 4);
    w.hA = (float*)take((int64_t)B * Nc * 512 * 4);
    w.hB = (float*)take((int64_t)B * Nc * 512 * 4);
    (void)e;
    w.total = off;
    return w;
}

}  // namespace

int fc_paconv_create(FcCursor& c, const int32_t* header, int n_header, fc_embedder* e) {
    if (n_header < 14) return FC_ERR_MODEL;
    if (header[12] != PA_K || header[13] != PA_M || e->d_in < 4) return FC_ERR_UNSUPPORTED;
    PaModel* pm = new (std::nothrow) PaModel();
    if (!pm) return FC_ERR_MODEL;
    pm->c_feat = e->d_in - 3;
    for (int i = 0; i < 4; ++i) {
        pm->sa[i].npoint = header[8 + i];
        if (pm->sa[i].npoint < 1) { delete pm; return FC_ERR_UNSUPPORTED; }
        for (int j = 0; j < 3; ++j) {
            PaLayer& L = pm->sa[i].layer[j];
            L.Cin = (j == 0) ? (i == 0 ? pm->c_feat : SA_W[i][0]) + 3 : SA_W[i][j];
            L.Cout = SA_W[i][j + 1];
            L.score = c.ptr(c.next(), PA_SCORE_FLOATS);
            L.lin = c.linear(PA_M * 2 * L.Cin, 0, L.Cout);
            if (!L.score) c.ok = false;
        }
    }
    for (int i = 0; i < 4; ++i) {
        pm->fp[i].n_layers = FP_N[i];
        pm->fp[i].Cin = FP_W[i][0] + (i == 0 ? pm->c_feat : 0);
        for (int j = 0; j < FP_N[i]; ++j)
            pm->fp[i].lin[j] = c.linear(j == 0 ? pm->fp[i].Cin : FP_W[i][j], 0, FP_W[i][j + 1]);
    }
    e->out_mlp = c.mlp(128, 0, e->out_hid, e->n_out_hid, e->E);
    e->paconv = pm;
    return FC_OK;
}

void fc_paconv_destroy(fc_embedder* e) { delete static_cast<PaModel*>(e->paconv); e->paconv = nullptr; }

int64_t fc_paconv_workspace_bytes(const fc_embedder* e, int B, int Nc) {
    const PaModel* pm = static_cast<const PaModel*>(e->paconv);
    if (!pm) return FC_ERR_MODEL;
    return carve_pa(e, pm, B, Nc, nullptr).total;
}

int fc_paconv_embed(const fc_embedder* e, const float* pts, float* out, int B, int Nc, void* ws, int64_t ws_bytes, int precision,
                    cudaStream_t s) {
    const PaModel* pm = static_cast<const PaModel*>(e->paconv);
    FC_REQUIRE(pm != nullptr);
    // npoint of every SA level is latched at pack time (the reference latches N//4 on its first call,
    // pointnet2_paconv_modules.py:37-38); a cloud must have at least that many points
    FC_REQUIRE(Nc > pm->sa[0].npoint && B <= 65535);
    PaWs w = carve_pa(e, pm, B, Nc, ws);
    if (w.total > ws_bytes) return FC_ERR_WORKSPACE;
    int rc;
    {
        const long long tot = (long long)B * Nc;
        split_points_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(pts, e->d_in, tot, w.xyz[0], w.feat[0], w.ldfeat[0]);
        fc_count_launch(); FC_LAUNCH_OK();
    }
    const int cfeat[5] = {pm->c_feat, 64, 128, 256, 512};
    for (int i = 0; i < 4; ++i) {
        const int n = w.n[i], m = w.n[i + 1];
        FC_REQUIRE(m <= n);
        rc = launch_fps(w.xyz[i], B, n, m, 0, w.fidx, w.xyz[i + 1], s);
        if (rc) return rc;
        rc = launch_knn_heap(w.xyz[i], w.xyz[i + 1], B, n, m, PA_K, w.kidx, nullptr, s);
        if (rc) return rc;
        const long long edges = (long long)B * m * PA_K;
        const int C0 = cfeat[i];
        int ldf = fc_round_up(3 + C0, 4);
        group_kernel<<<(unsigned)((edges + 127) / 128), 128, 0, s>>>(w.xyz[i], w.feat[i], w.ldfeat[i], C0, w.xyz[i + 1], w.kidx, n, m,
                                                                    edges, w.fA, ldf, w.dxyz);
        fc_count_launch(); FC_LAUNCH_OK();
        float* cur = w.fA; float* nxt = w.fB;
        for (int j = 0; j < 3; ++j) {
            const PaLayer& L = pm->sa[i].layer[j];
            const int ldx = PA_M * 2 * L.Cin;
            paconv_expand_kernel<<<(unsigned)(edges / PA_K), 256, 0, s>>>(cur, ldf, L.Cin, w.dxyz, L.score, w.X, ldx);
            fc_count_launch(); FC_LAUNCH_OK();
            GemmArgs g = fc_gemm_linear(L.lin, w.X, ldx, nxt, L.Cout, (int)edges, precision);
            g.act = FC_ACT_RELU;
            rc = fc_launch_gemm(g, s);
            if (rc) return rc;
            float* t = cur; cur = nxt; nxt = t;
            ldf = L.Cout;
        }
        const long long groups = (long long)B * m;
        const int Cout = pm->sa[i].layer[2].Cout;
        max_over_k_kernel<<<(unsigned)((groups * Cout + 255) / 256), 256, 0, s>>>(cur, ldf, Cout, groups, w.feat[i + 1], w.ldfeat[i + 1]);
        fc_count_launch(); FC_LAUNCH_OK();
    }
    // FP levels, deepest first: l_feat[i-1] = FP_i(l_xyz[i-1], l_xyz[i], l_feat[i-1], l_feat[i])
    const float* known_feat = w.feat[4]; int ldk = w.ldfeat[4]; int Ck = 512;
    float* fp_out[2] = {w.hA, w.hB};
    for (int lev = 3; lev >= 0; --lev) {
        const int n = w.n[lev], m = w.n[lev + 1];
        rc = launch_three_nn(w.xyz[lev], w.xyz[lev + 1], B, n, m, w.idx3, w.w3, nullptr, s);
        if (rc) return rc;
        const int C1 = cfeat[lev], Ct = Ck + C1, ldcat = fc_round_up(Ct, 4);
        const long long pts_tot = (long long)B * n;
        interp_concat_kernel<<<(unsigned)((pts_tot * Ct + 255) / 256), 256, 0, s>>>(known_feat, ldk, Ck, w.feat[lev], w.ldfeat[lev], C1,
                                                                                 w.idx3, w.w3, n, m, pts_tot, w.fpcat, ldcat);
        fc_count_launch(); FC_LAUNCH_OK();
        const PaFP& F = pm->fp[lev];
        FC_REQUIRE(F.Cin == Ct);
        const float* cur = w.fpcat; int ldc = ldcat;
        float* dst = nullptr;
        for (int j = 0; j < F.n_layers; ++j) {
            dst = (j == F.n_layers - 1) ? fp_out[lev & 1] : w.fph;
            if (dst == cur) dst = w.X;   // never in place
            GemmArgs g = fc_gemm_linear(F.lin[j], cur, ldc, dst, F.lin[j].N, (int)pts_tot, precision);
            g.act = FC_ACT_RELU;
            rc = fc_launch_gemm(g, s);
            if (rc) return rc;
            cur = dst; ldc = F.lin[j].N;
        }
        known_feat = cur; ldk = ldc; Ck = ldc;
    }
    // out MLP on the finest level (128 channels)
    FcMlpIn in{known_feat, ldk, nullptr, 0, nullptr, 0, 0};
    float* last = nullptr;
    float* bufA = (known_feat == w.hA) ? w.hB : w.hA;
    rc = fc_run_mlp_hidden(e->out_mlp, in, B * Nc, bufA, w.X, 512, precision, s, &last);
    if (rc) return rc;
    return fc_launch_gemm(fc_gemm_linear(e->out_mlp.out, last, 512, out, e->E, B * Nc, precision), s);
}

// ------------------------------------------------------------------------------------------ op-level C ABI (pointops)
extern "C" int fc_fps(const float* xyz, int B, int n, int m, int tie_block, int32_t* idx_out, float* new_xyz_out, fc_stream_t stream) {
    return launch_fps(xyz, B, n, m, tie_block, idx_out, new_xyz_out, (cudaStream_t)stream);
}
extern "C" int fc_knn_heap(const float* xyz, const float* new_xyz, int B, int n, int m, int k, int32_t* idx_out, float* dist2_out,
                           fc_stream_t stream) {
    return launch_knn_heap(xyz, new_xyz, B, n, m, k, idx_out, dist2_out, (cudaStream_t)stream);
}
extern "C" int fc_three_nn(const float* unknown, const float* known, int B, int n, int m, float* dist2_out, int32_t* idx_out,
                           fc_stream_t stream) {
    FC_REQUIRE(dist2_out != nullptr);
    return launch_three_nn(unknown, known, B, n, m, idx_out, nullptr, dist2_out, (cudaStream_t)stream);
}
extern "C" int fc_three_interpolate(const float* known_feat, int ldk, int C, const int32_t* idx, const float* weight, int B, int n, int m,
                                    float* out, int ldo, fc_stream_t stream) {
    FC_REQUIRE(known_feat && idx && weight && out && B > 0 && n > 0 && m > 0 && C > 0 && ldk >= C && ldo >= C);
    const long long pts = (long long)B * n;
    interp_concat_kernel<<<(unsigned)((pts * C + 255) / 256), 256, 0, (cudaStream_t)stream>>>(known_feat, ldk, C, nullptr, 0, 0, idx, weight,
                                                                                           n, m, pts, out, ldo);
    fc_count_launch(); FC_LAUNCH_OK();
    return FC_OK;
}
extern "C" int fc_group_points(const float* feat, int ldf, int C, const int32_t* idx, int B, int n, int m, int k, float* out, int ldo,
                               fc_stream_t stream) {
    FC_REQUIRE(feat && idx && out && B > 0 && n > 0 && m > 0 && k > 0 && C > 0 && ldf >= C && ldo >= C);
    const long long rows = (long long)B * m * k;
    gather_rows_kernel<<<(unsigned)((rows * C + 255) / 256), 256, 0, (cudaStream_t)stream>>>(feat, ldf, C, idx, n, (long long)m * k, rows, out, ldo);
    fc_count_launch(); FC_LAUNCH_OK();
    return FC_OK;
}
