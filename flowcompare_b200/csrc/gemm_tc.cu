// fp32-faithful GEMM on the 5th-gen tensor cores: 3xTF32 error-compensated tcgen05.mma with TMEM accumulators,
// operands staged by TMA (128B swizzle), the same fused epilogues as the FFMA kernel (gemm.cu).
//
//   C = A W^T  with  A = Ahi + Alo,  W = Whi + Wlo  (TF32 splits)   =>   D = Ahi Whi + Alo Whi + Ahi Wlo
// (the dropped Alo Wlo term is ~2^-22 relative).  W is split once at pack time.  A (an activation that only
// exists in fp32) is split ON CHIP and never touches HBM or shared memory again: TMA lands the raw fp32 tile in
// shared memory, each converter thread reads its own row (bank-conflict free under the 128B swizzle), rounds
// it to TF32 (hi) and keeps the exact remainder (lo), and writes both straight into TENSOR MEMORY
// (tcgen05.st), from where tcgen05.mma takes its A operand.  Only the B operand (the weights) is read from
// shared memory by the tensor core, which halves the shared-memory traffic per flop of the SS form.
//
// The tensor core truncates when it adds a product block to its accumulator (measured ~0.25 ulp one-sided per
// tcgen05.mma).  The two small compensation products therefore get their OWN accumulator (truncation at 2^-11
// of the magnitude), and the one GEMM whose output is the latent itself (ActNorm+LinearLU) applies its
// diagonal in fp32 in the epilogue (flow.cu), so the residual bias is below the fp32 noise of the reference.
//
// PERSISTENT kernel, one CTA per SM (18 warps, all 512 TMEM columns, ~225 KB of shared memory).  The CTA walks the
// list of 128 x BN output tiles (BN <= 96; N is cut into equal-ish multiples of 16, no padded columns) with stride
// gridDim.x.  The accumulators are DOUBLE BUFFERED in TMEM, so the epilogue of tile j runs while the tensor core is
// on tile j+1, and the TMA / converter / MMA pipelines never drain between tiles:
//   warp 0       TMA producer (one lane): 5 (3xTF32) or 6 (3xFP16) shared-memory stages of (A raw 16 KB, Whi, Wlo)
//   warp 1       TMEM allocator + MMA issuer (whole warp loops, one elected lane issues).  Issue is effectively
//                synchronous (the tensor queue is a couple of MMAs deep), so the warp PROBES the next stage's barriers
//                before it blocks in the issue and skips the wait when they have fired.  ONE issuer, in program
//                order: the accumulation order, and with it every output bit, is the same on every run (two issuer
//                warps sharing a k-block were 3-5 % faster on single GEMMs, equal on the whole step, and measurably
//                non-deterministic; one warp per accumulator was deterministic but 5 % slower).
//   warps 2-9    converters (two threads per tile row): fp32 smem row -> hi/lo -> tcgen05.st, published one step late
//                so the store latency overlaps the next split.  3xFP16: warps 2-5 take the even k-blocks, 6-9 the odd
//                ones (a thread converts its whole row); 3xTF32: each thread converts its half of every k-block
//   warps 10-17  epilogue (two warps per TMEM lane quadrant, alternate 16-column chunks): bias row prefetched while the
//                tile is still being accumulated; global traffic staged per warp through shared memory (16-byte
//                coalesced accesses)
// TMEM (512 columns): accumulator buffer b = [192b, 192b+96) main | [192b+96, 192b+192) compensation;
//                     [384,512) the A operand, in stages of HALF a k-block: hi columns then lo columns.
// Pipeline (mbarriers): full[s] (TMA bytes landed) -> converter -> conv[ts] (A k-block in TMEM) -> MMA ->
//   tcgen05.commit -> tfree[ts], w_free[s] (stage reusable), acc_full[b] -> epilogue -> acc_free[b].
// Measured on the way here (B200; numbers in DESIGN.md section 4): two CTAs per SM with single-buffered accumulators
// (the previous design: 372 -> 390 pairs/s going persistent), the barrier probe (+6 %), a branch-free GELU, hand TF32
// rounding and 16-byte staged stores (+23 %); dropped: a 4-accumulator split of the main product (no accuracy gain),
// TMA multicast of the weight tile over clusters of 2/4 and halving the weight bytes (no effect: not L2 bound), one
// N=2*BN MMA for Ahi*[Whi;Wlo], decoupled A/W rings, 64/80-wide tiles, all-warps converters, a staggered start.
#include <cuda_fp16.h>
#include "gemm.cuh"
#include "tcgen05.cuh"
#include <cuda.h>
#include <cstdio>
#include <atomic>
#include <mutex>
#include <unordered_map>

namespace {

constexpr int TC_BM = 128;
constexpr int TC_BK = 32;                      // 32 fp32 = one 128-byte swizzle row
constexpr int TC_STAGES = 5;                   // shared-memory stages: a load is issued 4 k-blocks of tensor time (~1.4 us) ahead
constexpr int TC_STAGES_F16 = 6;               // 3xFP16: a stage is 16 KB of A + 2 x 6 KB of W, tensor time per k-block is halved;
                                               // 7 fit, 6 leave room for the epilogue's residual prefetch tiles
constexpr int TC_BN_CAP = 96;                  // widest tile (accumulator width); 80 leaves room for 6 A stages (measured slower)
constexpr int TC_CONV_WARPS = 8;               // two converter threads per tile row (measured +10 % in 3xFP16 mode over one)
constexpr int TC_CONV_WARP0 = 2;               // first converter warp (any 4 consecutive warps cover the 4 TMEM lane quadrants)
constexpr int TC_EPI_WARP0 = TC_CONV_WARP0 + TC_CONV_WARPS;   // first epilogue warp
constexpr int TC_THREADS = 32 * (TC_EPI_WARP0 + 8);           // TMA, MMA issuer, converter warps, 8 epilogue warps
// Per operand format: F16 = false 3xTF32 (weights as fp32 TF32 hi/lo), true 3xFP16 (weights as fp16 hi / 2^11-scaled lo)
template <bool F16> struct TcCfg {
    static constexpr int STAGES = F16 ? TC_STAGES_F16 : TC_STAGES;
    static constexpr int W_ELT = F16 ? 2 : 4;                         // bytes per weight element in shared memory
    static constexpr int TS_COLS = F16 ? 16 : 32;                     // TMEM columns of one A stage (HALF a k-block: hi | lo)
    static constexpr int TSTAGES = (512 - 4 * TC_BN_CAP) / TS_COLS;   // TMEM stages of the A operand
    // stages x (16 KB A + Whi + Wlo at BN = 96) + 8 staging tiles of the epilogue + 1 KB alignment slack
    // 3xFP16 mode: the residual of an epilogue chunk arrives by cp.async one chunk ahead (the first chunk's before the
    // accumulator wait) in a second per-warp staging tile (two 2 KB swizzled tiles per epilogue warp)
    static constexpr bool RES_PF = F16;
    static constexpr int STG_FLOATS = F16 ? 1024 : 32 * 20;           // per-warp staging floats
    static constexpr int SMEM_BYTES = STAGES * (TC_BM * TC_BK * 4 + 2 * 96 * TC_BK * W_ELT) + 8 * STG_FLOATS * 4 + 1024;
};
constexpr int TC_A_BYTES = TC_BM * TC_BK * 4;  // 16 KB
constexpr int TC_TMEM_COLS = 512;                // one persistent CTA per SM
constexpr int TC_COL_ACC = 2 * TC_BN_CAP;      // accumulator buffer b: main at 192*b, compensation at 192*b + 96
constexpr int TC_COL_CORR = TC_BN_CAP;
constexpr int TC_COL_A = 4 * TC_BN_CAP;        // + TS_COLS * stage: first half hi, second half lo

struct TcParams {
    GemmArgs g;
    int BN;        // widest N tile of the launch (multiple of 16, <= TC_BN_CAP = 96)
    int T1, T2;    // k-blocks of segment 1 / 2
    int n_tiles, m_tiles;
    int tma_store; // STORE / LNQ epilogues: full 32 x 16 chunks leave through TMA stores (mapC) instead of per-thread stores
};

// ----------------------------------------------------------------------------- kernel
// One instantiation per (epilogue kind, activation, residual): with every variant inlined behind runtime branches the
// kernel was 80 KB of SASS and ncu showed an 88 % instruction-cache hit rate with "no instruction" among the top
// stall reasons of the epilogue warps.
//
// PERSISTENT: one CTA per SM walks the (m-tile, n-tile) list with stride gridDim.x.  The accumulators are double
// buffered in TMEM, so the epilogue of tile j (8 dedicated warps) runs while the tensor core is already on tile j+1;
// the TMA / converter / MMA pipelines never drain between tiles (global k-block counters carry the barrier phases).
template <int EPI, int ACT, bool RES, bool F16>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap mapA1, const __grid_constant__ CUtensorMap mapA2,
               const __grid_constant__ CUtensorMap mapWhi, const __grid_constant__ CUtensorMap mapWlo,
               const __grid_constant__ CUtensorMap mapC, const TcParams p) {
    constexpr int TC_STAGES = TcCfg<F16>::STAGES, TC_TSTAGES = TcCfg<F16>::TSTAGES, TS_COLS = TcCfg<F16>::TS_COLS;   // shadow the globals
    constexpr bool PARITY = F16;   // 3xFP16: the converter groups take turns on k-blocks
    extern __shared__ unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * TC_STAGES + 2 * TC_TSTAGES + 4];
    __shared__ uint32_t tmem_base_slot;
    __shared__ float ldj_sm[2][TC_BM];        // by tile parity: the only barrier between the two halves is the one inside a tile
    // the bias (and LayerNorm-q column sums) of the columns each epilogue warp handles in the current tile: chunk i of the warp
    // (columns half*16 + 32*i ..+15 of the tile) at [16*i ..+15].  Per warp, so the epilogue needs no CTA-wide barrier.
    __shared__ __align__(16) float bias_w[8][48];
    __shared__ __align__(16) float csum_w[8][48];

    const uint32_t raw = smem_u32(smem_raw);
    unsigned char* smem = smem_raw + ((1024u - (raw & 1023u)) & 1023u);   // SWIZZLE_128B tiles need 1024 B alignment
    const int BN = p.BN;                    // widest tile of this launch: shared-memory layout and TMA box
    const int w_box_bytes = BN * TC_BK * TcCfg<F16>::W_ELT;          // what one weight TMA box brings
    // 3xFP16: the Wlo box always sits 96 rows behind the Whi box (rows BN..95 of the slot are never written: they only feed
    // accumulator columns nobody reads), so that one MMA can run over [Whi; Wlo] whatever BN is
    const int w_bytes = F16 ? TC_BN_CAP * TC_BK * TcCfg<F16>::W_ELT : w_box_bytes;
    const int stage_bytes = TC_A_BYTES + 2 * w_bytes;
    auto a_raw = [&](int s) { return smem + s * stage_bytes; };
    auto w_hi = [&](int s) { return smem + s * stage_bytes + TC_A_BYTES; };
    auto w_lo = [&](int s) { return smem + s * stage_bytes + TC_A_BYTES + w_bytes; };
    float* stage_out = reinterpret_cast<float*>(smem + TC_STAGES * stage_bytes);   // 8 warps x [32][20] staging tiles
    uint64_t* full = bars;                                   // [TC_STAGES]  TMA bytes landed
    uint64_t* w_free = bars + TC_STAGES;                     // [TC_STAGES]  MMAs done reading the stage (A and W smem)
    uint64_t* conv = bars + 2 * TC_STAGES;                   // [TC_TSTAGES] A hi/lo written to TMEM
    uint64_t* tfree = bars + 2 * TC_STAGES + TC_TSTAGES;     // [TC_TSTAGES] MMAs done reading A TMEM
    uint64_t* acc_full = bars + 2 * TC_STAGES + 2 * TC_TSTAGES;   // [2] accumulators of a tile complete
    uint64_t* acc_free = acc_full + 2;                            // [2] epilogue has drained them (256 arrivals)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = p.T1 + p.T2;
    const int n_tiles = p.n_tiles, total_tiles = p.n_tiles * p.m_tiles;
    // N is cut into n_tiles tiles whose widths are multiples of 16 and differ by at most 16 (512 -> 96,96,80,80,80,80):
    // no padded columns go through the tensor core.  The TMA box stays BN rows (the extra rows are the next tile's).
    const int n_units = (p.g.N + 15) >> 4, n_base = n_units / n_tiles, n_rem = n_units % n_tiles;
    auto tile_n0_of = [&](int nt) { return 16 * (nt * n_base + min(nt, n_rem)); };
    auto tile_bn_of = [&](int nt) { return 16 * (n_base + (nt < n_rem ? 1 : 0)); };

    if (threadIdx.x == 0) {
        constexpr int CONV_GROUPS = PARITY ? 2 : 1;         // converter groups that take turns on k-blocks
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&w_free[s], 1); }
        for (int s = 0; s < TC_TSTAGES / 2; ++s) { mbar_init(&conv[s], 32 * 8 / CONV_GROUPS); mbar_init(&tfree[s], 1); }   // one pair per K-BLOCK of A in tensor memory
        for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_free[s], 32 * 8); }   // one arrival per thread
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "n"(TC_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_slot;

    if (warp == 0) {
        // ===================================================== TMA producer
        if (lane == 0) {
            uint32_t g = 0;   // k-blocks issued so far (all tiles)
            for (int L = blockIdx.x; L < total_tiles; L += gridDim.x) {
                const int n_tile = L % n_tiles, m0 = (L / n_tiles) * TC_BM;
                const int tile_n0 = tile_n0_of(n_tile);
                for (int t = 0; t < T; ++t, ++g) {
                    const int s = g % TC_STAGES;
                    const uint32_t ph = (g / TC_STAGES) & 1;
                    // the stage is free once its MMAs have retired: they imply that the converters finished reading its
                    // activation tile long before
                    mbar_wait(&w_free[s], ph ^ 1, 150 + t);
                    mbar_expect_tx(&full[s], (uint32_t)(TC_A_BYTES + 2 * w_box_bytes));
                    if (t < p.T1) tma_load_2d(&mapA1, a_raw(s), &full[s], t * TC_BK, m0);
                    else          tma_load_2d(&mapA2, a_raw(s), &full[s], (t - p.T1) * TC_BK, m0);
                    tma_load_2d(&mapWhi, w_hi(s), &full[s], t * TC_BK, tile_n0);
                    tma_load_2d(&mapWlo, w_lo(s), &full[s], t * TC_BK, tile_n0);
                }
            }
        }
    } else if (warp < TC_CONV_WARP0) {
        // ===================================================== MMA issuer
        // The whole warp runs the loop and ONE ELECTED lane issues: inside a divergent `if (lane == 0)` the compiler
        // cannot keep the descriptors in uniform registers and wraps every UTCHMMA in an ELECT/vote loop with R2UR moves.
        //
        // This warp is a serial program and MMA issue blocks (the tensor queue is a couple of MMAs deep), so everything it
        // does besides issuing is dead time for the tensor pipe.  Measured with knock-out builds (DESIGN.md section 4):
        // with NO MMAs, NO loads and NO conversion the loop still took ~780 cycles per k-block -- every mbarrier check
        // costs ~40 cycles, a commit ~30 -- against 288 tensor cycles for a 3xFP16 k-block.  Hence: ONE barrier per k-block
        // towards the converters (conv[]; it implies full[]: the converters only publish after they have seen the stage's
        // TMA bytes land, and the weights arrive on the same transaction barrier), one probe of the next one, two commits
        // (tfree[], w_free[]) and ring positions kept as counters (no division).
        int it = 0;
        bool conv_seen = false;   // the next k-block's barrier was seen complete by the probe
        int s = 0;                // shared-memory stage of the next k-block
        int ks = 0; uint32_t kph = 0;   // tensor-memory A stage (one per k-block) of the next k-block and its barrier phase
        for (int L = blockIdx.x; L < total_tiles; L += gridDim.x, ++it) {
            const int n_tile = L % n_tiles;
            const int tile_bn = tile_bn_of(n_tile);
            const int buf = it & 1;
            // instruction descriptor: D=f32 (bits 4-5 = 1), A=B=tf32 (2), K-major, N>>3 at bit 17, M>>4 at bit 24
            // (kind::f16: A = B = fp16 is format 0)
            const uint32_t idesc = (1u << 4) | ((F16 ? 0u : 2u) << 7) | ((F16 ? 0u : 2u) << 10) | ((uint32_t)(tile_bn >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            const uint32_t d_main = tmem + TC_COL_ACC * buf, d_corr = d_main + TC_COL_CORR;
            const uint32_t idesc_wide = (idesc & ~(0x3fu << 17)) | ((uint32_t)((TC_BN_CAP + tile_bn) >> 3) << 17);
            mbar_wait(&acc_free[buf], ((it >> 1) & 1) ^ 1, 190);     // the epilogue of tile it-2 has drained this buffer
            for (int t = 0; t < T; ++t) {
                if (!conv_seen) mbar_wait(&conv[ks], kph, 300 + t);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                {   // probe the NEXT k-block now: a wait after the issue is dead time for the tensor pipe
                    int kn = ks + 1; uint32_t pn = kph;
                    if (kn >= TC_TSTAGES / 2) { kn -= TC_TSTAGES / 2; pn ^= 1; }
                    conv_seen = mbar_test(&conv[kn], pn);
                }
                if (elect_one()) {
                    const uint64_t dbh = F16 ? make_kmajor_sw64_desc(smem_u32(w_hi(s))) : make_kmajor_sw128_desc(smem_u32(w_hi(s)));
                    const uint64_t dbl = F16 ? make_kmajor_sw64_desc(smem_u32(w_lo(s))) : make_kmajor_sw128_desc(smem_u32(w_lo(s)));
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        // the k-block's A operand: two half k-blocks of TS_COLS columns each (first half hi, second half lo)
                        const uint32_t t_hi = tmem + TC_COL_A + TS_COLS * (2 * ks + h), t_lo = t_hi + TS_COLS / 2;
                        if (F16) {
                            // one kind::f16 MMA covers the half k-block (16 k = 32 bytes of the 64-byte weight row).
                            // Whi and Wlo are adjacent 96-row boxes of the stage and the two accumulators adjacent 96-column
                            // blocks of TMEM: ONE MMA of N = 96 + tile_bn computes Ahi.[Whi; Wlo] -> [main | compensation].
                            // A TS-form kind::f16 MMA costs the same issue time at N = 192 as at N = 96
                            // (scripts/micro/peaks.cu), so two instructions per half k-block instead of three.
                            // (Columns tile_bn..95 of main receive the next tile's weight rows: never read.)
                            const uint64_t adv = (uint64_t)(h * 32 >> 4);
                            umma_f16_ts(d_main, t_hi, dbh + adv, idesc_wide, (t | h) != 0);
                            umma_f16_ts(d_corr, t_lo, dbh + adv, idesc, 1);               // (A - Ahi) 2^11 . Whi
                        } else {
#pragma unroll
                            for (int kk = 0; kk < 2; ++kk) {
                                const int k = 2 * h + kk;
                                const uint64_t adv = (uint64_t)(k * 32 >> 4);   // 8 tf32 = 32 bytes per k-step
                                umma_tf32_ts(d_corr, t_lo + 8 * kk, dbh + adv, idesc, (t | k) != 0);
                                umma_tf32_ts(d_corr, t_hi + 8 * kk, dbl + adv, idesc, 1);
                                umma_tf32_ts(d_main, t_hi + 8 * kk, dbh + adv, idesc, (t | k) != 0);
                            }
                        }
                    }
                    umma_commit(&tfree[ks]);                     // TMEM A stage reusable once these MMAs retire
                    umma_commit(&w_free[s]);                     // W smem stage reusable once these MMAs retire
                }
                __syncwarp();
                s = s + 1 == TC_STAGES ? 0 : s + 1;
                ks = ks + 1 == TC_TSTAGES / 2 ? 0 : ks + 1; if (ks == 0) kph ^= 1;
            }
            if (elect_one()) umma_commit(&acc_full[buf]);        // accumulators of this tile complete
            __syncwarp();
        }
    } else if (warp < TC_EPI_WARP0) {
        // ===================================================== converters: fp32 smem row -> (hi, lo) in TMEM
        const int quad = warp & 3;                   // TMEM lane quadrant this warp may touch
        const int row_in_tile = quad * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
        const int my_half = (warp - TC_CONV_WARP0) >> 2;   // 3xTF32: the first four warps take the first half of every k-block, the others the second
        // Software pipelined by one step: the tcgen05.st of a k-block (3xTF32: of a half) is in flight while the next one is
        // loaded and split; only then is it awaited and published (one arrival per thread on the k-block's conv[] barrier),
        // so the store latency is off the critical path.
        int s = 0; uint32_t sph = 0;   // shared-memory stage / phase of the current k-block
        int ks = 0; uint32_t kph = 0;  // tensor-memory A stage (one per k-block) / phase
        int pending = -1;              // k-block stage whose store has been issued but not yet published
        if constexpr (PARITY) {
            // Two converter groups take turns on k-blocks: every role of this kernel pays ~100 cycles per mbarrier wait (even on a
            // completed phase) plus the tcgen05.st round trip, so ONE group working through every k-block was a ~500-cycle serial
            // chain per k-block (knock-out builds: the pipeline ran at that pace with all the work removed).  A thread converts
            // its whole 32-float row of the k-block and writes it with one 32-column tcgen05.st.
            const int grp = (warp - TC_CONV_WARP0) >> 2;
            uint32_t g = 0;
            auto publish = [&]() {
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                mbar_arrive(&conv[pending]);
                pending = -1;
            };
            for (int L = blockIdx.x; L < total_tiles; L += gridDim.x) {
                for (int t = 0; t < T; ++t, ++g) {
                    if ((int)(g & 1) == grp) {
                        if (pending >= 0) publish();
                        mbar_wait(&full[s], sph, 400 + t);
                        const float4* rowp = reinterpret_cast<const float4*>(a_raw(s) + row_in_tile * 128);
                        uint32_t hl[32];   // [half 0: hi x8 | lo x8 | half 1: hi x8 | lo x8], two fp16 per column
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            // 128B swizzle: logical 16-byte chunk j of row r sits at physical chunk j ^ (r & 7); a quarter
                            // warp (8 consecutive rows) therefore hits all 32 banks exactly once
                            const float4 x = rowp[j ^ (row_in_tile & 7)];
                            const float xv[4] = {x.x, x.y, x.z, x.w};
                            const int base = 16 * (j >> 2) + 2 * (j & 3);
                            // hi = fp16(x) (11-bit significand, like TF32), lo = fp16((x - hi) * 2^11): the residual is
                            // taken from the value the tensor core will actually see, so fp16 subnormals lose nothing;
                            // |x| >= 65520 becomes inf and the row's result NaN (loud, never silently clipped)
#pragma unroll
                            for (int e = 0; e < 4; e += 2) {
                                const uint32_t hp = pack_f16x2(xv[e], xv[e + 1]);
                                float h0, h1;
                                unpack_f16x2(hp, h0, h1);
                                hl[base + (e >> 1)] = hp;
                                const float2 d2 = __fmul2_rn(__fadd2_rn(make_float2(xv[e], xv[e + 1]), make_float2(-h0, -h1)), make_float2(2048.0f, 2048.0f));
                                hl[base + 8 + (e >> 1)] = pack_f16x2(d2.x, d2.y);
                            }
                        }
                        mbar_wait(&tfree[ks], kph ^ 1, 450 + t);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        tmem_st32(tmem + lane_addr + TC_COL_A + TS_COLS * (2 * ks), hl);
                        pending = ks;
                    }
                    s = s + 1 == TC_STAGES ? 0 : s + 1; if (s == 0) sph ^= 1;
                    ks = ks + 1 == TC_TSTAGES / 2 ? 0 : ks + 1; if (ks == 0) kph ^= 1;
                }
            }
            if (pending >= 0) publish();
        } else
        for (int L = blockIdx.x; L < total_tiles; L += gridDim.x) {
            for (int t = 0; t < T; ++t) {
                if (pending >= 0) {      // never hold a finished stage back while waiting for the next k-block's data
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    mbar_arrive(&conv[pending]);
                    pending = -1;
                }
                mbar_wait(&full[s], sph, 400 + t);
                const float4* rowp = reinterpret_cast<const float4*>(a_raw(s) + row_in_tile * 128);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (h != my_half) continue;   // two threads per row: each converts its own half k-block
                    uint32_t hl[TS_COLS];   // this half k-block: first half hi, second half lo
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int j = 4 * h + jj;
                        const float4 x = rowp[j ^ (row_in_tile & 7)];   // 128B swizzle, as above
                        const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            // cvt.rna.tf32.f32 by hand (add half a TF32 ulp to the magnitude, clear the low 13 bits):
                            // 2 ALU ops instead of the 4 (add, inf test, select, mask) ptxas emits; inputs are finite
                            const uint32_t u = (__float_as_uint(xv[e]) + 0x1000u) & 0xffffe000u;
                            hl[4 * jj + e] = u;
                            hl[TS_COLS / 2 + 4 * jj + e] = __float_as_uint(xv[e] - __uint_as_float(u));
                        }
                    }
                    if (pending >= 0) {
                        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        mbar_arrive(&conv[pending]);
                    }
                    mbar_wait(&tfree[ks], kph ^ 1, 450 + t);   // the MMAs that read this TMEM stage have retired
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    tmem_st32(tmem + lane_addr + TC_COL_A + TS_COLS * (2 * ks + h), hl);
                    pending = ks;
                }
                s = s + 1 == TC_STAGES ? 0 : s + 1; if (s == 0) sph ^= 1;
                ks = ks + 1 == TC_TSTAGES / 2 ? 0 : ks + 1; if (ks == 0) kph ^= 1;
            }
        }
        if (pending >= 0) {
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(&conv[pending]);
        }
    } else {
        // ===================================================== epilogue (8 warps, 256 threads)
        // TMEM lane = row within the tile; the two warps of a quadrant take alternate 16-column chunks
        const int quad = warp & 3;
        const int row_in_tile = quad * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(quad * 32) << 16;
        const int ew = warp - TC_EPI_WARP0;          // 0..7
        const int half = ew >> 2;
        const int etid = threadIdx.x - 32 * TC_EPI_WARP0;   // 0..255
        const GemmArgs& a = p.g;
        // per-warp staging tile [32 rows][16 + 4 pad] (rows 16-byte aligned; a thread's own-row float4 accesses are
        // conflict free, the transposed ones 2-way at worst)
        float* stg = stage_out + ew * TcCfg<F16>::STG_FLOATS;
        int it = 0;
        bool tma_pending = false;
        for (int L = blockIdx.x; L < total_tiles; L += gridDim.x, ++it) {
            const int n_tile = L % n_tiles, m0 = (L / n_tiles) * TC_BM;
            const int tile_n0 = tile_n0_of(n_tile), tile_bn = tile_bn_of(n_tile);
            const int buf = it & 1;
            float* bias_sm = bias_w[ew];
            float* csum_sm = csum_w[ew];
            // while the tensor core is still on this tile: fetch its bias row (a cold L2 miss per 16-column chunk
            // otherwise -- measured ~600 cycles each) into shared memory
            const int last_row = min(m0 + TC_BM, a.M) - 1;
            const bool one_group = a.bias_group <= 0 || (m0 / a.bias_group) == (last_row / a.bias_group);
            const bool bias_smem = one_group && m0 < a.M;
            {
                const float* brow = a.bias;
                if (a.bias && a.bias_group > 0) brow = a.bias + (size_t)(m0 / a.bias_group) * a.bias_ld;
                __syncwarp();            // every lane is done with the previous tile's values
                for (int i = lane; i < 48; i += 32) {
                    const int ct = half * 16 + 32 * (i >> 4) + (i & 15);     // column within the tile
                    const int col = tile_n0 + ct;
                    const bool ok = ct < tile_bn && col < a.N;
                    bias_sm[i] = (brow && one_group && ok) ? brow[col] : 0.f;
                    csum_sm[i] = (EPI == FC_EPI_LNQ && ok) ? a.csum[col] : 0.f;
                }
            }
            // The residual of a chunk does not depend on the accumulator: its (L2-latency) loads are issued one chunk ahead,
            // and the first chunk's before the wait for the tensor core, so they overlap the mainloop / the previous chunk.
            const int row0 = m0 + quad * 32;
            const bool vec_base = row0 + 32 <= a.M && (a.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(a.C) & 15) == 0;
            const bool vec_res = RES && (a.ldres & 3) == 0 && (reinterpret_cast<uintptr_t>(a.res) & 15) == 0 &&
                                 (!a.res_scale || (reinterpret_cast<uintptr_t>(a.res_scale) & 15) == 0);
            // Prefetch (3xFP16, TMA-store launches): chunk c's residual is copied by cp.async into the staging tile the chunk's
            // output will later be written to (64B-swizzle layout, thread (r, q) -> row r, 16-byte slot q ^ ((r >> 1) & 3));
            // the two tiles alternate, so the copy for chunk c+1 runs while chunk c is computed and stored.
            const bool res_pf = TcCfg<F16>::RES_PF && RES && p.tma_store && vec_base && vec_res;
            int pb = 0;
            auto res_prefetch = [&](int c0n, int which) {
                const int coln = tile_n0 + c0n;
                // a chunk that straddles N (N a multiple of 4) is prefetched too: its 16-byte pieces beyond N are zero-filled
                // (src-size 0, nothing is read) and the TMA store clips them
                if (c0n < tile_bn && coln < a.N && (coln + 16 <= a.N || (a.N & 3) == 0)) {
                    const float* rp = a.res + (size_t)(row0 + (lane >> 2)) * a.ldres + coln + (lane & 3) * 4;
                    const uint32_t dst0 = smem_u32(stg + which * 512);
                    const uint32_t nbytes = coln + (lane & 3) * 4 < a.N ? 16u : 0u;
                    if (nbytes == 0u) rp = a.res;     // keep the (unused) address in bounds
    #pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int rr = (lane >> 2) + 8 * i;
                        const uint32_t dst = dst0 + (uint32_t)(rr * 64 + ((((lane & 3) ^ ((rr >> 1) & 3))) << 4));
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(dst), "l"(rp + (nbytes ? (size_t)(8 * i) * a.ldres : (size_t)0)), "r"(nbytes) : "memory");
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            if (res_pf) {
                if (tma_pending) {       // the last chunk of the previous tile may still be read by its TMA store
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    tma_pending = false;
                    __syncwarp();
                }
                res_prefetch(half * 16, pb);
            }
            // Same for the coupling epilogue's latent values (8 per row and chunk): copied ahead into a compact [32][12] tile
            // behind the [32][20] staging tile.
            const bool cpl_pf = TcCfg<F16>::RES_PF && EPI == FC_EPI_COUPLING && row0 + 32 <= a.M &&
                                ((a.ldx | a.col0) & 1) == 0 && (reinterpret_cast<uintptr_t>(a.x) & 7) == 0;
            auto cpl_prefetch = [&](int c0n) {
                const int coln = tile_n0 + c0n;
                if (c0n < tile_bn && coln + 16 <= a.N) {
                    const float* gx = a.x + (size_t)(row0 + (lane >> 2)) * a.ldx + a.col0 + (coln >> 1) + (lane & 3) * 2;
                    const uint32_t dst0 = smem_u32(stg + 640 + (lane >> 2) * 12 + (lane & 3) * 2);
    #pragma unroll
                    for (int i = 0; i < 4; ++i)
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(dst0 + (uint32_t)(8 * i * 12 * 4)), "l"(gx + (size_t)(8 * i) * a.ldx) : "memory");
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            if (cpl_pf) cpl_prefetch(half * 16);
            float mu = 0.f, rstd = 0.f;
            if (EPI == FC_EPI_LNQ && m0 + row_in_tile < a.M) { mu = a.row_mu[m0 + row_in_tile]; rstd = a.row_rstd[m0 + row_in_tile]; }
            mbar_wait(&acc_full[buf], (it >> 1) & 1, 500);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            __syncwarp();                                      // bias_sm / csum_sm visible to the whole warp
            const uint32_t acc_main = tmem + lane_addr + TC_COL_ACC * buf, acc_corr = acc_main + TC_COL_CORR;
            const int row = m0 + row_in_tile;
            const bool row_ok = row < a.M;
            const int n0 = tile_n0;
            float ldj = 0.f;
            const float* bias_row = a.bias;
            if (a.bias && a.bias_group > 0 && row_ok) bias_row = a.bias + (size_t)(row / a.bias_group) * a.bias_ld;
            // the accumulator loads of chunk c+1 are in flight while chunk c goes through its bias / activation / stores
            uint32_t r[16], rc[16];
            if (half * 16 < tile_bn) tmem_ld16x2_issue(acc_main + (uint32_t)(half * 16), acc_corr + (uint32_t)(half * 16), r, rc);
            for (int c0 = half * 16; c0 < tile_bn; c0 += 32) {
                float v[16];
                if (tma_pending) {       // the previous chunk's TMA store must have READ the staging tile before it is rewritten
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    tma_pending = false;
                }
                __syncwarp();
                tmem_ld16x2_wait(r, rc);
    #pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    const float2 m2 = make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1]));
                    const float2 c2 = make_float2(__uint_as_float(rc[j]), __uint_as_float(rc[j + 1]));
                    const float2 o2 = F16 ? __ffma2_rn(c2, make_float2(4.8828125e-4f, 4.8828125e-4f), m2) : __fadd2_rn(m2, c2);
                    v[j] = o2.x; v[j + 1] = o2.y;
                }
                if (c0 + 32 < tile_bn) tmem_ld16x2_issue(acc_main + (uint32_t)(c0 + 32), acc_corr + (uint32_t)(c0 + 32), r, rc);
                const int col = n0 + c0;
                if (col >= a.N) continue;                     // warp-uniform
                if (EPI == FC_EPI_LNQ) {
    #pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (col + j < a.N) v[j] = rstd * (v[j] - mu * csum_sm[(c0 >> 5) * 16 + j]) + bias_sm[(c0 >> 5) * 16 + j];
                } else if (bias_row && bias_smem) {
                    // four 16-byte broadcast loads (bias_sm is 16-byte aligned and c0 a multiple of 16); zero beyond N
    #pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 b4 = *reinterpret_cast<const float4*>(bias_sm + (c0 >> 5) * 16 + 4 * q);
                        const float2 s0 = __fadd2_rn(make_float2(v[4 * q], v[4 * q + 1]), make_float2(b4.x, b4.y));
                        const float2 s1 = __fadd2_rn(make_float2(v[4 * q + 2], v[4 * q + 3]), make_float2(b4.z, b4.w));
                        v[4 * q] = s0.x; v[4 * q + 1] = s0.y; v[4 * q + 2] = s1.x; v[4 * q + 3] = s1.y;
                    }
                } else if (bias_row) {
                    if (col + 15 < a.N && ((reinterpret_cast<uintptr_t>(bias_row + col) & 15) == 0)) {
                        // four 16-byte loads at a warp-uniform address (issued back to back) instead of 16 predicated ones
                        const float4* b4 = reinterpret_cast<const float4*>(bias_row + col);
                        const float4 b0 = __ldg(b4), b1 = __ldg(b4 + 1), b2 = __ldg(b4 + 2), b3 = __ldg(b4 + 3);
                        v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
                        v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
                        v[8] += b2.x; v[9] += b2.y; v[10] += b2.z; v[11] += b2.w;
                        v[12] += b3.x; v[13] += b3.y; v[14] += b3.z; v[15] += b3.w;
                    } else {
    #pragma unroll
                        for (int j = 0; j < 16; ++j) if (col + j < a.N) v[j] += bias_row[col + j];
                    }
                }
                if (EPI == FC_EPI_STORE || EPI == FC_EPI_LNQ) {
                    // Global traffic goes through a per-warp staging tile so that it is COALESCED: with one thread per
                    // row, direct loads/stores touch 32 different lines per instruction (ncu: the residual layers took 2x
                    // as long as the plain ones).  Each warp instruction below moves 2 rows x 64 contiguous bytes.
                    const int sr = lane >> 4, sc = lane & 15;
                    // fast path (every full interior chunk): 16-byte accesses, 8 rows x 64 B per warp instruction, no
                    // per-element predicates or address arithmetic -- the scalar form below cost ~19 instructions per
                    // element, more than the GELU
                    const bool vec = vec_base && col + 16 <= a.N;
                    // TMA-store launches also take a chunk that straddles N through the fast path (the store clips it)
                    const bool vect = vec || (vec_base && p.tma_store && (a.N & 3) == 0 && (!RES || res_pf));
                    const int r8 = lane >> 2, c4 = (lane & 3) * 4;
                    float4* my_row4 = reinterpret_cast<float4*>(stg + lane * 20);
                    if (RES) {
                        if (vect && res_pf) {
                            asm volatile("cp.async.wait_group 0;" ::: "memory");
                            __syncwarp();
                            const unsigned char* rb = reinterpret_cast<const unsigned char*>(stg + pb * 512) + lane * 64;
                            const int sw = (lane >> 1) & 3;
    #pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float4 rv = *reinterpret_cast<const float4*>(rb + ((q ^ sw) << 4));
                                if (a.res_scale) {
                                    const float4 rs = col + 4 * q < a.N ? *reinterpret_cast<const float4*>(a.res_scale + col + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
                                    v[4 * q] = fmaf(rs.x, rv.x, v[4 * q]); v[4 * q + 1] = fmaf(rs.y, rv.y, v[4 * q + 1]);
                                    v[4 * q + 2] = fmaf(rs.z, rv.z, v[4 * q + 2]); v[4 * q + 3] = fmaf(rs.w, rv.w, v[4 * q + 3]);
                                } else {
                                    const float2 s0 = __fadd2_rn(make_float2(v[4 * q], v[4 * q + 1]), make_float2(rv.x, rv.y));
                                    const float2 s1 = __fadd2_rn(make_float2(v[4 * q + 2], v[4 * q + 3]), make_float2(rv.z, rv.w));
                                    v[4 * q] = s0.x; v[4 * q + 1] = s0.y; v[4 * q + 2] = s1.x; v[4 * q + 3] = s1.y;
                                }
                            }
                            res_prefetch(c0 + 32, pb ^ 1);   // the other tile: its last TMA store was waited for at the top of this chunk
                        } else if (vec && vec_res) {
                            const float* rp = a.res + (size_t)(row0 + r8) * a.ldres + col + c4;
                            float4 rx4[4];
    #pragma unroll
                            for (int i = 0; i < 4; ++i) rx4[i] = __ldg(reinterpret_cast<const float4*>(rp + (size_t)(8 * i) * a.ldres));
    #pragma unroll
                            for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(stg + (r8 + 8 * i) * 20 + c4) = rx4[i];
                            __syncwarp();
    #pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float4 rv = my_row4[q];
                                if (a.res_scale) {
                                    const float4 rs = *reinterpret_cast<const float4*>(a.res_scale + col + 4 * q);
                                    v[4 * q] = fmaf(rs.x, rv.x, v[4 * q]); v[4 * q + 1] = fmaf(rs.y, rv.y, v[4 * q + 1]);
                                    v[4 * q + 2] = fmaf(rs.z, rv.z, v[4 * q + 2]); v[4 * q + 3] = fmaf(rs.w, rv.w, v[4 * q + 3]);
                                } else {
                                    v[4 * q] += rv.x; v[4 * q + 1] += rv.y; v[4 * q + 2] += rv.z; v[4 * q + 3] += rv.w;
                                }
                            }
                            __syncwarp();
                        } else {
                            float rx[16];   // all loads first, then all shared stores: no store->load ordering stalls
    #pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const int gr = row0 + 2 * i + sr;
                                rx[i] = (gr < a.M && col + sc < a.N) ? __ldg(a.res + (size_t)gr * a.ldres + col + sc) : 0.f;
                            }
    #pragma unroll
                            for (int i = 0; i < 16; ++i) stg[(2 * i + sr) * 20 + sc] = rx[i];
                            __syncwarp();
    #pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const float rv = stg[lane * 20 + j];
                                if (col + j < a.N) v[j] = a.res_scale ? fmaf(a.res_scale[col + j], rv, v[j]) : v[j] + rv;
                            }
                            __syncwarp();
                        }
                    }
                    if (ACT == FC_ACT_GELU) {
    #pragma unroll
                        for (int j = 0; j < 16; j += 2) {
                            const float2 g2 = fc_gelu_erf_fast2(make_float2(v[j], v[j + 1]));
                            v[j] = g2.x; v[j + 1] = g2.y;
                        }
                    } else if (ACT == FC_ACT_LRELU) {
    #pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = fc_leaky_relu02(v[j]);
                    } else if (ACT == FC_ACT_RELU) {
    #pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
                    }
                    if (vect && p.tma_store) {
                        // The chunk as a 32-row x 64-byte tile in the 64B-swizzle layout (16-byte chunk q of row r at q ^ ((r >> 1) & 3):
                        // every thread writes its own row conflict free), handed to the TMA unit by one lane: no transposed
                        // shared-memory reads, no per-thread global stores or address arithmetic (UTMASTG).
                        float* stile = stg + (res_pf ? pb * 512 : 0);
                        unsigned char* sb = reinterpret_cast<unsigned char*>(stile) + lane * 64;
                        const int sw = (lane >> 1) & 3;
    #pragma unroll
                        for (int q = 0; q < 4; ++q)
                            *reinterpret_cast<float4*>(sb + ((q ^ sw) << 4)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(&mapC, stile, col, row0);
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                        tma_pending = true;
                        pb ^= 1;
                        continue;
                    }
    #pragma unroll
                    for (int q = 0; q < 4; ++q) my_row4[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                    __syncwarp();
                    if (vec) {
                        float* gp = a.C + (size_t)(row0 + r8) * a.ldc + col + c4;
                        float4 ox4[4];
    #pragma unroll
                        for (int i = 0; i < 4; ++i) ox4[i] = *reinterpret_cast<const float4*>(stg + (r8 + 8 * i) * 20 + c4);
    #pragma unroll
                        for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(gp + (size_t)(8 * i) * a.ldc) = ox4[i];
                    } else {
                        float ox[16];
    #pragma unroll
                        for (int i = 0; i < 16; ++i) ox[i] = stg[(2 * i + sr) * 20 + sc];
    #pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const int gr = row0 + 2 * i + sr;
                            if (gr < a.M && col + sc < a.N) a.C[(size_t)gr * a.ldc + col + sc] = ox[i];
                        }
                    }
                    __syncwarp();
                } else if (EPI == FC_EPI_KVSPLIT && a.kv_f16) {
                    // the same for the 3xFP16 attention: fp16 hi and fp16 (x - hi); k rows are 128 bytes, v^T rows kv_ncp halfs
                    uint32_t hp[8], lp[8];      // packed pairs (columns 2j, 2j+1)
                    __half hh[16], lh[16];
    #pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        hh[j] = __float2half_rn(v[j]);
                        lh[j] = __float2half_rn(v[j] - __half2float(hh[j]));
                    }
    #pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        hp[j] = (uint32_t)__half_as_ushort(hh[2 * j]) | ((uint32_t)__half_as_ushort(hh[2 * j + 1]) << 16);
                        lp[j] = (uint32_t)__half_as_ushort(lh[2 * j]) | ((uint32_t)__half_as_ushort(lh[2 * j + 1]) << 16);
                    }
                    if (col < 64) {
                        // k: a row's 16 values are 32 contiguous bytes; staged so that a warp instruction writes 8 rows x 32 B
                        uint32_t* stw = reinterpret_cast<uint32_t*>(stg);
                        const int r8 = lane >> 2, part = lane & 3;
    #pragma unroll
                        for (int pass = 0; pass < 2; ++pass) {
                            __half* dstbase = reinterpret_cast<__half*>(pass == 0 ? a.C : a.kv_klo);
                            uint4* my = reinterpret_cast<uint4*>(stw + lane * 20);
                            my[0] = pass == 0 ? make_uint4(hp[0], hp[1], hp[2], hp[3]) : make_uint4(lp[0], lp[1], lp[2], lp[3]);
                            my[1] = pass == 0 ? make_uint4(hp[4], hp[5], hp[6], hp[7]) : make_uint4(lp[4], lp[5], lp[6], lp[7]);
                            __syncwarp();
    #pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int gr = row0 + r8 + 8 * i;
                                if (gr < a.M)
                                    *reinterpret_cast<uint2*>(dstbase + (size_t)gr * 64 + col + 4 * part) =
                                        *reinterpret_cast<const uint2*>(stw + (r8 + 8 * i) * 20 + 2 * part);
                            }
                            __syncwarp();
                        }
                    } else if (row_ok) {
                        const int bcl = row / a.kv_nc, key = row - bcl * a.kv_nc;
                        __half* th = reinterpret_cast<__half*>(a.kv_vthi) + ((size_t)bcl * 64 + (col - 64)) * a.kv_ncp + key;
                        __half* tl = reinterpret_cast<__half*>(a.kv_vtlo) + ((size_t)bcl * 64 + (col - 64)) * a.kv_ncp + key;
    #pragma unroll
                        for (int j = 0; j < 16; ++j) { th[(size_t)j * a.kv_ncp] = hh[j]; tl[(size_t)j * a.kv_ncp] = lh[j]; }
                    }
                } else if (EPI == FC_EPI_KVSPLIT) {
                    // to_kv feeding the tcgen05 attention (attention_tc.cu): TF32 hi/lo copies, v transposed per cloud.
                    // BN = 64, so N-tile 0 is k and N-tile 1 is v.
                    float lo16[16];
    #pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float h = __uint_as_float((__float_as_uint(v[j]) + 0x1000u) & 0xffffe000u);
                        lo16[j] = v[j] - h;
                        v[j] = h;
                    }
                    if (col < 64) {
                        // k: rows stay rows; two staged, coalesced 16-byte passes (hi, then lo)
                        const int r8 = lane >> 2, c4 = (lane & 3) * 4;
                        float4* my_row4 = reinterpret_cast<float4*>(stg + lane * 20);
    #pragma unroll
                        for (int pass = 0; pass < 2; ++pass) {
                            float* dstbase = pass == 0 ? a.C : a.kv_klo;
    #pragma unroll
                            for (int q = 0; q < 4; ++q)
                                my_row4[q] = pass == 0 ? make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3])
                                                       : make_float4(lo16[4 * q], lo16[4 * q + 1], lo16[4 * q + 2], lo16[4 * q + 3]);
                            __syncwarp();
    #pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int gr = row0 + r8 + 8 * i;
                                if (gr < a.M)
                                    *reinterpret_cast<float4*>(dstbase + (size_t)gr * 64 + col + c4) =
                                        *reinterpret_cast<const float4*>(stg + (r8 + 8 * i) * 20 + c4);
                            }
                            __syncwarp();
                        }
                    } else if (row_ok) {
                        // v: transposed; the 32 lanes of a warp hold 32 consecutive keys -> each store instruction writes
                        // one contiguous run per cloud
                        const int bcl = row / a.kv_nc, key = row - bcl * a.kv_nc;
                        float* th = a.kv_vthi + ((size_t)bcl * 64 + (col - 64)) * a.kv_ncp + key;
                        float* tl = a.kv_vtlo + ((size_t)bcl * 64 + (col - 64)) * a.kv_ncp + key;
    #pragma unroll
                        for (int j = 0; j < 16; ++j) { th[(size_t)j * a.kv_ncp] = v[j]; tl[(size_t)j * a.kv_ncp] = lo16[j]; }
                    }
                } else if (EPI == FC_EPI_COUPLING && row0 + 32 <= a.M && col + 16 <= a.N &&
                           ((a.ldx | a.col0) & 1) == 0 && (reinterpret_cast<uintptr_t>(a.x) & 7) == 0) {
                    // reference models/affine_coupling.py:40-46.  Interior chunk of a full 32-row quadrant: the chunk's 8 latent
                    // values per row go through the warp's staging tile so that the global accesses are COALESCED (a warp
                    // instruction moves 8 rows x 32 contiguous bytes; one thread per row touched 32 different sectors per
                    // instruction and every sector twice: the latent accesses were 4.7 % of the whole GEMM class)
                    const int r8 = lane >> 2, c2 = (lane & 3) * 2;
                    float* gx = a.x + (size_t)(row0 + r8) * a.ldx + a.col0 + (col >> 1) + c2;
                    float2 lx[4];
                    float4* my4 = reinterpret_cast<float4*>(stg + lane * 20);
                    float4 xa, xb;
                    if (cpl_pf) {
                        asm volatile("cp.async.wait_group 0;" ::: "memory");
                        __syncwarp();
                        const float4* pf4 = reinterpret_cast<const float4*>(stg + 640 + lane * 12);
                        xa = pf4[0]; xb = pf4[1];
                        __syncwarp();
                        cpl_prefetch(c0 + 32);
                    } else {
    #pragma unroll
                        for (int i = 0; i < 4; ++i) lx[i] = *reinterpret_cast<const float2*>(gx + (size_t)(8 * i) * a.ldx);
    #pragma unroll
                        for (int i = 0; i < 4; ++i) *reinterpret_cast<float2*>(stg + (r8 + 8 * i) * 20 + c2) = lx[i];
                        __syncwarp();
                        xa = my4[0]; xb = my4[1];
                    }
                    float xs[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
    #pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float sig = 1.0f / (1.0f + expf(-v[2 * q]));
                        const float sc = (2.0f * sig - 1.0f) + 1.0f;
                        xs[q] = fmaf(xs[q], sc, v[2 * q + 1]);
                        ldj += logf(sc);
                    }
                    my4[0] = make_float4(xs[0], xs[1], xs[2], xs[3]);
                    my4[1] = make_float4(xs[4], xs[5], xs[6], xs[7]);
                    __syncwarp();
    #pragma unroll
                    for (int i = 0; i < 4; ++i) lx[i] = *reinterpret_cast<const float2*>(stg + (r8 + 8 * i) * 20 + c2);
    #pragma unroll
                    for (int i = 0; i < 4; ++i) *reinterpret_cast<float2*>(gx + (size_t)(8 * i) * a.ldx) = lx[i];
                    __syncwarp();
                } else if (!row_ok) {
                    // nothing: out-of-range rows of the coupling / augment epilogues
                } else if (EPI == FC_EPI_COUPLING) {
                    // reference models/affine_coupling.py:40-46 (see gemm.cu for the arithmetic notes)
                    float* xrow = a.x + (size_t)row * a.ldx + a.col0 + (col >> 1);
                    if (col + 16 <= a.N && (reinterpret_cast<uintptr_t>(xrow) & 7) == 0) {
                        // interior chunk: the row's 8 latent values move as four 8-byte accesses, loads first
                        float2 xv[4];
    #pragma unroll
                        for (int q = 0; q < 4; ++q) xv[q] = *reinterpret_cast<const float2*>(xrow + 2 * q);
    #pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float sig0 = 1.0f / (1.0f + expf(-v[4 * q]));
                            const float sc0 = (2.0f * sig0 - 1.0f) + 1.0f;
                            const float sig1 = 1.0f / (1.0f + expf(-v[4 * q + 2]));
                            const float sc1 = (2.0f * sig1 - 1.0f) + 1.0f;
                            xv[q].x = fmaf(xv[q].x, sc0, v[4 * q + 1]);
                            xv[q].y = fmaf(xv[q].y, sc1, v[4 * q + 3]);
                            ldj += logf(sc0);
                            ldj += logf(sc1);
                        }
    #pragma unroll
                        for (int q = 0; q < 4; ++q) *reinterpret_cast<float2*>(xrow + 2 * q) = xv[q];
                    } else {
    #pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            if (col + 2 * q + 1 < a.N) {
                                const float sig = 1.0f / (1.0f + expf(-v[2 * q]));
                                const float sc = (2.0f * sig - 1.0f) + 1.0f;
                                float* xp = xrow + q;
                                *xp = fmaf(*xp, sc, v[2 * q + 1]);
                                ldj += logf(sc);
                            }
                        }
                    }
                } else if (EPI == FC_EPI_COUPLING_INV) {
                    // reference models/affine_coupling.py:48-62 (sampling pass): x2 = (y2 - t) / s
    #pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        if (col + 2 * q + 1 < a.N) {
                            const float sig = 1.0f / (1.0f + expf(-v[2 * q]));
                            const float sc = (2.0f * sig - 1.0f) + 1.0f;
                            float* xp = a.x + (size_t)row * a.ldx + a.col0 + (col >> 1) + q;
                            *xp = (*xp - v[2 * q + 1]) / sc;
                        }
                    }
                } else if (EPI == FC_EPI_AUGMENT) {
                    // reference models/distributions.py:128-153 + models/augmenter.py:49-63
    #pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        if (col + 2 * q + 1 < a.N) {
                            const int j = (col >> 1) + q;
                            const float e = a.eps[(size_t)row * a.ld_eps + j];
                            a.x[(size_t)row * a.ldx + a.col0 + j] = fmaf(expf(v[2 * q + 1]), e, v[2 * q]);
                            ldj += fmaf(0.5f * e, e, v[2 * q + 1]) + 0.91893853320467274178f;
                        }
                    }
                }
            }
            if (EPI == FC_EPI_COUPLING || EPI == FC_EPI_AUGMENT) {
                // the two threads that share a row combine their partial log-dets in a fixed order (deterministic)
                // (measured: reading the old partial before the accumulator wait, a per-quadrant barrier and releasing the
                // accumulator before this tail made the coupling launches 7 % SLOWER, 300 vs 281 us)
                if (half == 1) ldj_sm[buf][row_in_tile] = ldj;
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (half == 0 && row_ok) {
                    const float tot = ldj + ldj_sm[buf][row_in_tile];
                    float* pp = a.part + (size_t)n_tile * a.M + row;
                    if (EPI == FC_EPI_COUPLING) *pp += tot; else *pp = tot;
                }
            }
            // this thread's TMEM reads of the tile are complete (every tcgen05.ld above is followed by its wait)
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(&acc_free[buf]);
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");    // this warp's TMA stores have landed
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TC_TMEM_COLS));
    }
}

// ----------------------------------------------------------------------------- host: tensor maps
struct MapKey {
    const void* base; uint64_t inner, outer, stride; uint32_t box_outer; int f16;
    bool operator==(const MapKey& o) const {
        return base == o.base && inner == o.inner && outer == o.outer && stride == o.stride && box_outer == o.box_outer && f16 == o.f16;
    }
};
struct MapKeyHash {
    size_t operator()(const MapKey& k) const {
        size_t h = std::hash<const void*>()(k.base);
        h ^= std::hash<uint64_t>()(k.inner * 1315423911u + k.outer) + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
        h ^= std::hash<uint64_t>()(k.stride * 31 + k.box_outer * 2 + k.f16) + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
        return h;
    }
};
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;
std::mutex g_maps_mu;

// [outer][inner] row-major with row stride `stride_floats` ELEMENTS; box = 32 x box_outer, OOB -> 0.  fp32 elements with
// the 128B swizzle (a box row is 128 bytes) or, f16 = 1, fp16 elements with the 64B swizzle (a box row is 64 bytes).
// Maps only encode address + geometry, so they are cached (the flow re-uses the same workspace every call).
bool get_map(const void* base, uint64_t inner, uint64_t outer, uint64_t stride_floats, uint32_t box_outer, CUtensorMap* out,
             int f16 = 0) {
    MapKey key{base, inner, outer, stride_floats, box_outer, f16};
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *out = it->second; return true; }
    FcEncodeTiledFn enc = fc_get_encode_fn();
    if (!enc) return false;
    cuuint64_t dims[2] = {inner, outer};
    // f16 = 2: the OUTPUT map of the TMA-store epilogue: fp32, boxes of 16 columns (64 bytes) x box_outer rows, 64B swizzle
    cuuint64_t strides[1] = {stride_floats * (f16 == 1 ? 2 : 4)};
    cuuint32_t box[2] = {(cuuint32_t)(f16 == 2 ? 16 : TC_BK), box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUtensorMap m;
    CUresult r = enc(&m, f16 == 1 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims,
                     strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, f16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                     f16 == 2 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        fprintf(stderr, "flowcompare_b200: cuTensorMapEncodeTiled failed (%d): base=%p inner=%llu outer=%llu stride=%llu box=%ux%u\n",
                (int)r, (const void*)base, (unsigned long long)inner, (unsigned long long)outer,
                (unsigned long long)stride_floats, (unsigned)TC_BK, box_outer);
        return false;
    }
    if (g_maps.size() > 65536) g_maps.clear();
    g_maps.emplace(key, m);
    *out = m;
    return true;
}

}  // namespace

bool fc_gemm_tc_supported(const GemmArgs& a) {
    if (!a.Whi || !a.Wlo || a.ldk <= 0) return false;
    if ((a.lda1 & 3) || (reinterpret_cast<uintptr_t>(a.A1) & 15)) return false;
    if (a.K2 && ((a.lda2 & 3) || (reinterpret_cast<uintptr_t>(a.A2) & 15))) return false;
    if ((reinterpret_cast<uintptr_t>(a.Whi) & 15) || (reinterpret_cast<uintptr_t>(a.Wlo) & 15)) return false;
    if (a.M < 1 || a.N < 16) return false;
    return true;
}

namespace {
template <int EPI, int ACT, bool RES, bool F16>
cudaError_t launch_tc2(cudaLaunchConfig_t cfg, int dev, const CUtensorMap& mA1, const CUtensorMap& mA2, const CUtensorMap& mWh,
                       const CUtensorMap& mWl, const CUtensorMap& mC, const TcParams& p) {
    // the dynamic shared-memory opt-in is PER DEVICE (and per instantiation): one bit per device id
    static std::atomic<uint64_t> configured{0};
    const uint64_t bit = 1ull << (dev & 63);
    if (!(configured.load(std::memory_order_acquire) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<EPI, ACT, RES, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             TcCfg<F16>::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        configured.fetch_or(bit, std::memory_order_release);
    }
    cfg.dynamicSmemBytes = TcCfg<F16>::SMEM_BYTES;
    return cudaLaunchKernelEx(&cfg, gemm_tc_kernel<EPI, ACT, RES, F16>, mA1, mA2, mWh, mWl, mC, p);
}
template <int EPI, int ACT, bool RES>
cudaError_t launch_tc(const cudaLaunchConfig_t& cfg, int dev, int f16, const CUtensorMap& mA1, const CUtensorMap& mA2,
                      const CUtensorMap& mWh, const CUtensorMap& mWl, const CUtensorMap& mC, const TcParams& p) {
    return f16 ? launch_tc2<EPI, ACT, RES, true>(cfg, dev, mA1, mA2, mWh, mWl, mC, p)
               : launch_tc2<EPI, ACT, RES, false>(cfg, dev, mA1, mA2, mWh, mWl, mC, p);
}
int sm_count(int dev) {   // per device, cached
    static std::atomic<int> cache[64];
    int v = cache[dev & 63].load(std::memory_order_relaxed);
    if (!v) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return 0;
        cache[dev & 63].store(v, std::memory_order_relaxed);
    }
    return v;
}
}  // namespace

int fc_launch_gemm_tc(const GemmArgs& a, cudaStream_t stream) {
    FC_REQUIRE(fc_gemm_tc_supported(a));
    if (a.epi == FC_EPI_STORE || a.epi == FC_EPI_LNQ) FC_REQUIRE(a.C != nullptr);
    if (a.epi == FC_EPI_LNQ) FC_REQUIRE(a.row_mu && a.row_rstd && a.csum && a.bias && a.bias_group == 0);
    if (a.epi == FC_EPI_COUPLING || a.epi == FC_EPI_AUGMENT) FC_REQUIRE(a.x && a.part && (a.N % 2) == 0);
    if (a.epi == FC_EPI_COUPLING_INV) FC_REQUIRE(a.x && (a.N % 2) == 0);
    if (a.epi == FC_EPI_KVSPLIT)
        FC_REQUIRE(a.N == 128 && fc_tc_bn(a.N) == 64 && a.C && a.kv_klo && a.kv_vthi && a.kv_vtlo && a.kv_nc > 0 &&
                   a.kv_ncp >= a.kv_nc && (reinterpret_cast<uintptr_t>(a.C) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(a.kv_klo) & 15) == 0);
    TcParams p;
    p.g = a;
    p.BN = fc_tc_bn(a.N);
    p.T1 = fc_tc_kpad(a.K1) / TC_BK;
    p.T2 = a.K2 ? fc_tc_kpad(a.K2) / TC_BK : 0;
    FC_REQUIRE(p.BN <= TC_BN_CAP && (p.BN & 15) == 0);
    FC_REQUIRE(a.ldk == (p.T1 + p.T2) * TC_BK);
    p.n_tiles = fc_tc_n_tiles(a.N);
    p.m_tiles = (a.M + TC_BM - 1) / TC_BM;
    CUtensorMap mA1, mA2, mWh, mWl;
    if (!get_map(a.A1, (uint64_t)a.K1, (uint64_t)a.M, (uint64_t)a.lda1, TC_BM, &mA1)) return FC_ERR_CUDA;
    if (a.K2) { if (!get_map(a.A2, (uint64_t)a.K2, (uint64_t)a.M, (uint64_t)a.lda2, TC_BM, &mA2)) return FC_ERR_CUDA; }
    else mA2 = mA1;
    const int f16 = a.tc_fmt ? 1 : 0;
    if (!get_map(a.Whi, (uint64_t)a.ldk, (uint64_t)p.n_tiles * p.BN, (uint64_t)a.ldk, (uint32_t)p.BN, &mWh, f16)) return FC_ERR_CUDA;
    if (!get_map(a.Wlo, (uint64_t)a.ldk, (uint64_t)p.n_tiles * p.BN, (uint64_t)a.ldk, (uint32_t)p.BN, &mWl, f16)) return FC_ERR_CUDA;
    // TMA-store epilogue: plain-store epilogues whose output rows are 16-byte aligned
    CUtensorMap mC = mA1;
    p.tma_store = 0;
    if ((a.epi == FC_EPI_STORE || a.epi == FC_EPI_LNQ) && (a.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(a.C) & 15) == 0) {
        if (!get_map(a.C, (uint64_t)a.N, (uint64_t)a.M, (uint64_t)a.ldc, 32, &mC, 2)) return FC_ERR_CUDA;
        p.tma_store = 1;
    }
    int dev = 0;
    FC_CUDA_OK(cudaGetDevice(&dev));
    const int nsm = sm_count(dev);
    FC_REQUIRE(nsm > 0);
    const int total_tiles = p.n_tiles * p.m_tiles;
    FcProfScope prof(FC_CLS_GEMM_TC, 2.0 * a.M * a.N * (a.K1 + a.K2),
                     4.0 * ((double)a.M * (a.K1 + a.K2) + (double)a.N * (a.K1 + a.K2) + (double)a.M * a.N), stream,
                     (long long)(a.K1 + a.K2) | ((long long)a.N << 16) | ((long long)a.epi << 32) | ((long long)a.act << 36) |
                         ((long long)(a.res != nullptr) << 40));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(total_tiles < nsm ? total_tiles : nsm);      // persistent: one CTA per SM
    cfg.blockDim = dim3(TC_THREADS);
    cfg.stream = stream;
    const bool res = a.res != nullptr;
    cudaError_t le = cudaErrorInvalidValue;
    if (a.epi == FC_EPI_STORE) {
        if (a.act == FC_ACT_NONE)       le = res ? launch_tc<FC_EPI_STORE, FC_ACT_NONE, true>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p)
                                                 : launch_tc<FC_EPI_STORE, FC_ACT_NONE, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
        else if (a.act == FC_ACT_GELU)  le = res ? launch_tc<FC_EPI_STORE, FC_ACT_GELU, true>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p)
                                                 : launch_tc<FC_EPI_STORE, FC_ACT_GELU, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
        else if (a.act == FC_ACT_LRELU) le = res ? launch_tc<FC_EPI_STORE, FC_ACT_LRELU, true>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p)
                                                 : launch_tc<FC_EPI_STORE, FC_ACT_LRELU, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
        else if (a.act == FC_ACT_RELU)  le = res ? launch_tc<FC_EPI_STORE, FC_ACT_RELU, true>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p)
                                                 : launch_tc<FC_EPI_STORE, FC_ACT_RELU, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
    } else if (a.epi == FC_EPI_LNQ && a.act == FC_ACT_NONE && !res) {
        le = launch_tc<FC_EPI_LNQ, FC_ACT_NONE, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
    } else if (a.epi == FC_EPI_COUPLING) {
        le = launch_tc<FC_EPI_COUPLING, FC_ACT_NONE, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
    } else if (a.epi == FC_EPI_AUGMENT) {
        le = launch_tc<FC_EPI_AUGMENT, FC_ACT_NONE, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
    } else if (a.epi == FC_EPI_COUPLING_INV) {
        le = launch_tc<FC_EPI_COUPLING_INV, FC_ACT_NONE, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
    } else if (a.epi == FC_EPI_KVSPLIT && a.act == FC_ACT_NONE && !res) {
        le = launch_tc<FC_EPI_KVSPLIT, FC_ACT_NONE, false>(cfg, dev, f16, mA1, mA2, mWh, mWl, mC, p);
    } else {
        return FC_ERR_UNSUPPORTED;
    }
    FC_CUDA_OK(le);
    fc_count_launch();
    FC_LAUNCH_OK();
    return FC_OK;
}
