// DGCNN context embedders: `DGCNNembedder.forward` (reference models/pytorch_gcn.py:81-107) and
// `DGCNNembedderGlobal.forward` (:143-188).
//
// Per EdgeConv block: kNN in feature space (knn.cu) -> one per-POINT GEMM producing [P | Q]
// (gemm.cu; eval-mode BatchNorm folded into the weights at pack time) -> gather-max + LeakyReLU
// (edgeconv.cu), written straight into its column slice of the [B*Nc, 512] concat buffer that conv5
// consumes, so `torch.cat((x1,x2,x3,x4))` (pytorch_gcn.py:102) never happens.
#include "model.cuh"
#include <new>
#include <cstring>

int fc_paconv_create(FcCursor& c, const int32_t* header, int n_header, fc_embedder* e);
void fc_paconv_destroy(fc_embedder* e);
int64_t fc_paconv_workspace_bytes(const fc_embedder* e, int B, int Nc);
int fc_paconv_embed(const fc_embedder* e, const float* pts, float* out, int B, int Nc, void* ws, int64_t ws_bytes,
                    int precision, cudaStream_t s);

namespace {

// pooled[b] = [max_n y[b,n,:] | mean_n y[b,n,:]]   (reference pytorch_gcn.py:178-181)
__global__ void pool_max_mean_kernel(const float* __restrict__ y, int ldy, int N, int C, float* __restrict__ pooled) {
    const int b = blockIdx.y;
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int part = threadIdx.x >> 5, nparts = blockDim.x >> 5;
    __shared__ float smax[8][33];
    __shared__ float ssum[8][33];
    float mx = -INFINITY, sm = 0.f;
    if (c < C)
        for (int n = part; n < N; n += nparts) {
            const float v = y[((size_t)b * N + n) * ldy + c];
            mx = fmaxf(mx, v); sm += v;
        }
    smax[part][threadIdx.x & 31] = mx; ssum[part][threadIdx.x & 31] = sm;
    __syncthreads();
    if (part == 0 && c < C) {
        for (int p = 1; p < nparts; ++p) { mx = fmaxf(mx, smax[p][threadIdx.x & 31]); sm += ssum[p][threadIdx.x & 31]; }
        pooled[(size_t)b * 2 * C + c] = mx;
        pooled[(size_t)b * 2 * C + C + c] = sm / (float)N;
    }
}

struct EmbWs {
    float *feat, *pq, *hA, *hB, *pooled, *norms; int32_t* idx;
    int64_t total_bytes;
};

EmbWs carve_emb_ws(const fc_embedder* e, int B, int Nc, void* base) {
    EmbWs w{};
    const int64_t M = (int64_t)B * Nc;
    int64_t off = 0;
    auto take = [&](int64_t bytes) { char* p = base ? reinterpret_cast<char*>(base) + off : nullptr;
                                     off += fc_round_up_ll(bytes, 256); return p; };
    w.feat = (float*)take(M * 512 * 4);
    w.pq = (float*)take(M * 512 * 4);
    w.hA = (float*)take(M * 512 * 4);
    w.hB = (float*)take(M * 512 * 4);
    w.pooled = (float*)take((int64_t)B * 1024 * 4);
    w.idx = (int32_t*)take(M * e->k * 4);
    w.norms = (float*)take(fc_knn_scratch_floats(B, Nc, Nc, true) * 4);
    w.total_bytes = off;
    return w;
}

}  // namespace

extern "C" int fc_embedder_create(const int32_t* header, int n_header, const int64_t* table, int n_table,
                                  const float* arena, int64_t arena_floats, fc_embedder** out) {
    FC_REQUIRE(header && table && arena && out && n_header >= 8);
    if (header[0] != FC_EMB_MAGIC || (header[1] != FC_ARENA_VERSION && header[1] != FC_ARENA_VERSION_F16)) return FC_ERR_MODEL;
    if (reinterpret_cast<uintptr_t>(arena) & 15) return FC_ERR_MODEL;
    fc_embedder* e = new (std::nothrow) fc_embedder();
    if (!e) return FC_ERR_MODEL;
    e->kind = header[2]; e->d_in = header[3]; e->k = header[4]; e->E = header[5];
    e->out_hid = header[6]; e->n_out_hid = header[7];
    e->arena = arena; e->arena_floats = arena_floats;
    FcCursor c{table, n_table, 0, arena, arena_floats, true};
    c.tc_fmt = header[1] == FC_ARENA_VERSION_F16 ? 1 : 0;
    if (e->kind == 0 || e->kind == 1) {
        if (e->k < 1 || e->k > 64 || e->out_hid > 512 || e->d_in < 1) { delete e; return FC_ERR_UNSUPPORTED; }
        const int cin[4] = {e->d_in, 64, 64, 128};
        const int cout[4] = {64, 64, 128, 256};
        for (int i = 0; i < 4; ++i) {
            e->ec[i].Cin = cin[i]; e->ec[i].Cout = cout[i];
            e->ec[i].pq = c.linear(cin[i], 0, 2 * cout[i]);
        }
        e->conv5 = c.linear(512, 0, 512);
        e->out_mlp = c.mlp(e->kind == 1 ? 1024 : 512, 0, e->out_hid, e->n_out_hid, e->E);
    } else if (e->kind == 2) {
        int rc = fc_paconv_create(c, header, n_header, e);
        if (rc) { delete e; return rc; }
    } else { delete e; return FC_ERR_UNSUPPORTED; }
    if (!c.ok || c.pos != n_table) { fc_embedder_destroy(e); return FC_ERR_MODEL; }
    *out = e;
    return FC_OK;
}

extern "C" void fc_embedder_destroy(fc_embedder* e) {
    if (!e) return;
    if (e->kind == 2) fc_paconv_destroy(e);
    delete e;
}

extern "C" int64_t fc_embedder_workspace_bytes(const fc_embedder* e, int B, int Nc) {
    if (!e || B <= 0 || Nc <= 0) return FC_ERR_INVALID_ARG;
    if (e->kind == 2) return fc_paconv_workspace_bytes(e, B, Nc);
    return carve_emb_ws(e, B, Nc, nullptr).total_bytes;
}

extern "C" int fc_embed(const fc_embedder* e, const float* pts, float* out, int B, int Nc, int32_t* knn_idx_out,
                        void* workspace, int64_t workspace_bytes, int precision, fc_stream_t stream_) {
    FC_REQUIRE(e && pts && out && B > 0 && Nc > 0);
    cudaStream_t s = (cudaStream_t)stream_;
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return FC_ERR_WORKSPACE;
    if (e->kind == 2) return fc_paconv_embed(e, pts, out, B, Nc, workspace, workspace_bytes, precision, s);
    FC_REQUIRE(Nc >= e->k);
    EmbWs w = carve_emb_ws(e, B, Nc, workspace);
    if (w.total_bytes > workspace_bytes) return FC_ERR_WORKSPACE;
    const int M = B * Nc;
    const int col[4] = {0, 64, 128, 256};
    int rc;
    for (int i = 0; i < 4; ++i) {
        const float* xin = (i == 0) ? pts : w.feat + col[i - 1];
        const int ldin = (i == 0) ? e->d_in : 512;
        int32_t* idx = knn_idx_out ? knn_idx_out + (size_t)i * M * e->k : w.idx;
        rc = fc_knn_launch(xin, ldin, (long long)Nc * ldin, xin, ldin, (long long)Nc * ldin, B, Nc, Nc, e->ec[i].Cin,
                           e->k, 0, idx, nullptr, w.norms, s);
        if (rc) return rc;
        // the kNN is bit-exact by contract and its input feeds a discrete decision, so the [P|Q] GEMM
        // always runs in exact fp32
        rc = fc_launch_gemm(fc_gemm_linear(e->ec[i].pq, xin, ldin, w.pq, 512, M, 0), s);
        if (rc) return rc;
        rc = fc_launch_edgeconv_gather_max(w.pq, 512, idx, B, Nc, e->k, e->ec[i].Cout, w.feat + col[i], 512, s);
        if (rc) return rc;
    }
    GemmArgs g5 = fc_gemm_linear(e->conv5, w.feat, 512, w.pq, 512, M, 0);
    g5.act = FC_ACT_LRELU;
    rc = fc_launch_gemm(g5, s);
    if (rc) return rc;
    if (e->kind == 0) {
        FcMlpIn in{w.pq, 512, nullptr, 0, nullptr, 0, 0};
        float* last = nullptr;
        rc = fc_run_mlp_hidden(e->out_mlp, in, M, w.hA, w.hB, 512, precision, s, &last);
        if (rc) return rc;
        return fc_launch_gemm(fc_gemm_linear(e->out_mlp.out, last, 512, out, e->E, M, precision), s);
    }
    pool_max_mean_kernel<<<dim3(512 / 32, B), 256, 0, s>>>(w.pq, 512, Nc, 512, w.pooled);
    fc_count_launch();
    FC_LAUNCH_OK();
    FcMlpIn in{w.pooled, 1024, nullptr, 0, nullptr, 0, 0};
    float* last = nullptr;
    rc = fc_run_mlp_hidden(e->out_mlp, in, B, w.hA, w.hB, 512, 0, s, &last);
    if (rc) return rc;
    return fc_launch_gemm(fc_gemm_linear(e->out_mlp.out, last, 512, out, e->E, B, 0), s);
}
