"""CPU checks of constants / index arithmetic that live inside the CUDA sources (no GPU, no library calls):
the branch-free GELU's polynomial and the N-tile partition of the tcgen05 GEMM."""
import math
import os
import re

import numpy as np

from flowcompare_b200 import packing

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gelu_coefficients():
    src = open(os.path.join(ROOT, "flowcompare_b200", "csrc", "common.cuh")).read()
    body = src[src.index("float fc_gelu_erf_fast(float x)"):]
    body = body[:body.index("return")]
    clamp = float(re.search(r"fminf\(fabsf\(x\), ([0-9.eE+-]+)f\)", body).group(1))
    first = float(re.search(r"float r = ([0-9.eE+-]+)f;", body).group(1))
    rest = [float(v) for v in re.findall(r"r = fmaf\(r, u, ([0-9.eE+-]+)f\);", body)]
    return clamp, [first] + rest


def test_fast_gelu_polynomial_matches_exact_gelu():
    """fp32 emulation of fc_gelu_erf_fast (csrc/common.cuh): relu(x) - |x| * 2^(u r(u) - 1) vs 0.5 x (1 + erf(x/sqrt2))."""
    clamp, coef = _gelu_coefficients()
    assert len(coef) == 8 and 6.0 < clamp < 7.0
    x = np.linspace(-12.0, 12.0, 400001).astype(np.float32)
    u = np.minimum(np.abs(x), np.float32(clamp))
    r = np.full_like(u, np.float32(coef[0]))
    for c in coef[1:]:
        r = r * u + np.float32(c)
    e = np.exp2((r * u - np.float32(1.0)).astype(np.float64))
    got = -np.abs(x).astype(np.float64) * e + np.maximum(x, 0).astype(np.float64)
    want = np.array([0.5 * v * (1.0 + math.erf(v / math.sqrt(2.0))) for v in x.astype(np.float64)])
    assert np.abs(got - want).max() < 1e-7


def _tiles(N, bnmax=96):
    """Mirror of gemm_tc.cu: n_tiles = ceil(N / bnmax); widths are multiples of 16 that differ by at most 16."""
    n_tiles = (N + bnmax - 1) // bnmax
    units = (N + 15) // 16
    base, rem = divmod(units, n_tiles)
    n0 = [16 * (t * base + min(t, rem)) for t in range(n_tiles)]
    bn = [16 * (base + (1 if t < rem else 0)) for t in range(n_tiles)]
    return n0, bn


def test_gemm_tile_partition_covers_n_without_padding_columns():
    for N in (16, 64, 96, 100, 128, 256, 300, 512, 588, 1024, 97, 193):
        n0, bn = _tiles(N)
        assert len(bn) == packing.tc_n_tiles(N)
        assert max(bn) <= packing.tc_bn(N) <= 96 and min(bn) >= 16 and all(b % 16 == 0 for b in bn)
        assert max(bn) - min(bn) <= 16
        assert n0[0] == 0 and all(n0[i] + bn[i] == n0[i + 1] for i in range(len(bn) - 1))
        assert n0[-1] + bn[-1] == (N + 15) // 16 * 16                    # exactly N rounded up to 16: no padded tile columns
        # the TMA box is tc_bn(N) rows from n0: it must stay inside the packed weight rows (n_tiles * tc_bn)
        assert n0[-1] + packing.tc_bn(N) <= packing.tc_n_tiles(N) * packing.tc_bn(N)


def _tc_source():
    return open(os.path.join(ROOT, "flowcompare_b200", "csrc", "gemm_tc.cu")).read()


def _tc_define(name):
    m = re.search(r"constexpr int %s\s*=\s*([^;]+);" % name, _tc_source())
    assert m, name
    return m.group(1).strip()


def test_fused_whi_wlo_mma_tmem_layout_and_smem_budget():
    """3xFP16 (gemm_tc.cu): ONE tcgen05.mma of N = TC_BN_CAP + tile_bn runs over the adjacent [Whi; Wlo] boxes of a stage and
    lands in the adjacent [main | compensation] accumulators.  The layout facts that makes legal, checked against the source's
    constants: the compensation accumulator sits exactly TC_BN_CAP columns behind the main one, every wide N is a legal UMMA
    shape for M = 128 (multiple of 16, <= 256) and fits the 6-bit N field of the instruction descriptor, the wide write stays
    inside its own accumulator buffer (below the next buffer and the A-operand stages), and the Wlo slot starts on a whole
    8-row swizzle atom of the 64-byte fp16 weight rows so that one descriptor walks both boxes."""
    cap = int(_tc_define("TC_BN_CAP"))
    bk = int(_tc_define("TC_BK"))
    src = _tc_source()
    # the fp16 issue path is the fused one: the wide descriptor carries N = TC_BN_CAP + tile_bn, and the MMA that uses it
    # writes from the main accumulator on, so that its upper TC_BN_CAP columns land in the compensation accumulator
    assert re.search(r"idesc_wide = \(idesc & ~\(0x3fu << 17\)\) \| \(\(uint32_t\)\(\(TC_BN_CAP \+ tile_bn\) >> 3\) << 17\);", src)
    assert re.search(r"umma_f16_ts\(d_main, t_hi, dbh \+ adv, idesc_wide,", src)
    assert "umma_f16_ts(d_corr, t_hi, dbl" not in src            # no separate Ahi.Wlo MMA (the unfused three-MMA form)
    assert _tc_define("TC_COL_CORR").replace(" ", "") == "TC_BN_CAP"
    assert _tc_define("TC_COL_ACC").replace(" ", "") == "2*TC_BN_CAP"
    assert _tc_define("TC_COL_A").replace(" ", "") == "4*TC_BN_CAP"
    col_acc, col_a = 2 * cap, 4 * cap
    assert col_a <= 512 - 4 * 16                       # at least four 16-column A stages remain in the 512 TMEM columns
    for N in (64, 128, 256, 300, 512, 588):
        _, bn = _tiles(N, cap)
        for b in bn:
            wide = cap + b
            assert wide % 16 == 0 and 16 <= wide <= 256
            assert (wide >> 3) < 64
            assert wide <= col_acc                      # [main | compensation[0:b)] never reaches accumulator buffer 1 or the A stages
    row_bytes = bk * 2                                  # fp16 weights: 64-byte rows, SWIZZLE_64B atoms of 8 rows = 512 B
    assert (cap * row_bytes) % (8 * row_bytes) == 0
    # shared memory of the launch (TcCfg<true>::SMEM_BYTES: stages sized for 96-row boxes whatever BN is) fits the 227 KB opt-in
    stages = int(_tc_define("TC_STAGES_F16"))
    assert re.search(r"static constexpr int STAGES = F16 \? TC_STAGES_F16 : TC_STAGES;", src)
    stg_floats = int(re.search(r"static constexpr int STG_FLOATS = F16 \? (\d+) :", src).group(1))
    smem = stages * (128 * bk * 4 + 2 * cap * bk * 2) + 8 * stg_floats * 4 + 1024
    assert smem <= 227 * 1024


def test_error_compensated_operand_schemes_reach_fp32_accuracy():
    """The arithmetic the tensor-core GEMM relies on, with the product's own pack-time splits (packing.f16_split / tf32_round):
    D = Ahi.Whi + 2^-11 (Alo.Whi + Ahi.Wlo) for 3xFP16 (hi = fp16(x), lo = fp16((x - hi) 2^11)) and
    D = Ahi.Whi + Alo.Whi + Ahi.Wlo for 3xTF32, products and sums taken exactly (fp64) so that only the OPERAND scheme is
    measured: both must be as close to the exact product as an fp32 GEMM is (~K^0.5 2^-24 relative to |a||w| per term; the
    dropped Alo.Wlo term is 2^-22 of a term).  A plain single fp16 / TF32 product is shown to be 1000x worse."""
    import torch
    g = torch.Generator().manual_seed(0)
    M, N, K = 64, 48, 512
    A = torch.randn(M, K, generator=g)
    W = torch.randn(N, K, generator=g) / math.sqrt(K)
    exact = A.double() @ W.double().t()
    fp32 = (A @ W.t()).double()
    e_fp32 = (fp32 - exact).abs().max().item()
    ah, al = packing.f16_split(A)
    wh, wl = packing.f16_split(W)
    d16 = ah.double() @ wh.double().t() + (al.double() @ wh.double().t() + ah.double() @ wl.double().t()) / 2048.0
    e16 = (d16 - exact).abs().max().item()
    single16 = (ah.double() @ wh.double().t() - exact).abs().max().item()
    a_hi = packing.tf32_round(A); a_lo = packing.tf32_round(A - a_hi)
    w_hi = packing.tf32_round(W); w_lo = packing.tf32_round(W - w_hi)
    d32 = a_hi.double() @ w_hi.double().t() + a_lo.double() @ w_hi.double().t() + a_hi.double() @ w_lo.double().t()
    e32 = (d32 - exact).abs().max().item()
    assert e16 < 2e-6 and e32 < 2e-6, (e16, e32)
    assert e16 < 4 * e_fp32 + 1e-7 and e32 < 4 * e_fp32 + 1e-7, (e16, e32, e_fp32)        # as good as an fp32 GEMM
    assert single16 > 200 * e16                                                           # what the compensation buys
    # range: the hi part overflows exactly where the docs say (|x| >= 65520 -> inf), lo stays clear of fp16 subnormals for normal x
    assert torch.isinf(packing.f16_split(torch.tensor([65520.0]))[0]).all()
    x = torch.tensor([1.0 + 2.0 ** -12, 3.14159265, 1e-3])
    hi, lo = packing.f16_split(x)
    rec = hi.double() + lo.double() / 2048.0
    assert ((rec - x.double()).abs() / x.double()).max().item() < 2.0 ** -21


def test_knn_select_algorithm_model_matches_plain_sort_incl_masses_of_ties():
    """tests/knn_select_sim.py (a lane-by-lane model of knn_select_kernel) against a plain (key desc, index asc) sort: random
    rows of one and several segments, k = 1 / 40 / 64, rows shorter than a warp, exact pairs of duplicates, and MASSES of equal
    keys -- the exact-bisection path of the kernel (more than SEL_CAP survivors), incl. ties that straddle segments and the
    carried list, whose index order no GPU test compares with the oracle on more than pairs."""
    from tests import knn_select_sim as sim
    rng = np.random.RandomState(0)
    stats = {}
    cases = []
    for nt, k in [(33, 1), (40, 40), (100, 7), (1250, 40), (1280, 64), (1281, 40), (3000, 40), (2048, 64)]:
        cases.append((rng.randn(nt).astype(np.float32), k))
    dup = rng.randn(625).astype(np.float32)
    cases.append((np.concatenate([dup, dup]), 40))                                   # every key twice
    cases.append((np.zeros(1500, np.float32), 64))                                   # all equal
    cases.append((rng.choice(np.array([-1.0, 0.5, 2.0], np.float32), 2000), 40))     # three values: masses of ties at the threshold
    few = rng.randn(3000).astype(np.float32); few[rng.rand(3000) < 0.6] = 7.0         # 60 % share the LARGEST key, 3 segments
    cases.append((few, 64))
    low = rng.randn(2600).astype(np.float32); low[rng.rand(2600) < 0.9] = -3.0        # 90 % share a key BELOW the top-k
    cases.append((low, 40))
    mix = np.round(rng.randn(4000) * 2).astype(np.float32)                           # ~15 distinct values, 4 segments
    cases.append((mix, 40))
    for keys, k in cases:
        got = sim.select(keys, k, stats)
        want = sim.reference(keys, k)
        assert np.array_equal(got, want), (len(keys), k, got[:8], want[:8])
    assert stats.get("compaction", 0) > 0 and stats.get("bisection", 0) > 0          # both paths of the kernel were exercised
