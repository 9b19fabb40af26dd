"""GPU tests of the op-level pointops entry points (fc_fps / fc_knn_heap / fc_three_nn / fc_three_interpolate /
fc_group_points, through flowcompare_b200.pointops -> ctypes -> C ABI) against

  * the REFERENCE's own compiled kernels (oracle/_ref/libpointops_ref.so: the reference's unmodified
    lib/pointops/src/*/*_cuda_kernel.cu built by oracle/build_ref_pointops.sh) -- bit-exact indices, and
  * the CPU restatement oracle/pointops_ref.c (which the PAConv goldens were generated with), so that restatement is
    pinned to the compiled reference too.

The reference library is built from the reference's source tree, which is not part of the repository; without it the
reference comparisons are skipped.  test_outputs_equal_pinned_digests then still catches any change of these kernels' outputs,
against this project's own pinned outputs (tests/pointops_cases.py; not reference data).
"""
import time

import pytest
import torch

from flowcompare_b200 import configs, pointops as fpo, spec
from oracle import pointops_refcuda as ref
from oracle import port_paconv
from tests import pointops_cases as pc
from tests.pointops_cases import FPS_CASES, KNN_CASES, NN_CASES

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
needs_ref = pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libpointops_ref.so not built (needs /root/reference once)")
_cloud = pc.cloud


@needs_ref
@pytest.mark.parametrize("B,n,m,dup", FPS_CASES)
def test_fps_bit_exact_vs_reference_kernel(B, n, m, dup):
    x = pc.fps_inputs(B, n, m, dup)
    want = ref.furthestsampling(x, m)
    got, nx = fpo.furthestsampling(x, m, return_xyz=True)
    assert torch.equal(got, want)
    assert torch.equal(nx, torch.gather(x, 1, got.long().unsqueeze(-1).expand(-1, -1, 3)))


@pytest.mark.parametrize("B,n,m,dup", FPS_CASES[:4] + FPS_CASES[6:7])
def test_fps_matches_cpu_restatement(B, n, m, dup):
    x = _cloud(B, n, n + m, dup)
    assert torch.equal(fpo.furthestsampling(x.to(DEV), m).cpu(), port_paconv.furthestsampling(x, m))


def test_fps_lowest_index_tie_rule():
    """tie_block < 0: greedy farthest point where equal distances (exact duplicates) go to the LOWEST index."""
    import numpy as np
    x = _cloud(1, 2500, 5, duplicates=True)
    got = fpo.furthestsampling(x.to(DEV), 600, tie_block=-1).cpu()[0].tolist()
    xc = x[0].numpy()
    d = np.full(2500, 1e10, dtype=np.float32)
    old, want = 0, [0]
    for _ in range(599):
        dx = (xc - xc[old]).astype(np.float32)
        # fmaf(dz, dz, fmaf(dy, dy, dx * dx)) emulated through float64 (products of two floats are exact there)
        t = (dx[:, 0] * dx[:, 0]).astype(np.float32)
        t = (dx[:, 1].astype(np.float64) * dx[:, 1] + t).astype(np.float32)
        t = (dx[:, 2].astype(np.float64) * dx[:, 2] + t).astype(np.float32)
        d = np.minimum(d, t)
        old = int(np.argmax(d))          # first maximum = lowest index
        want.append(old)
    assert got == want


@needs_ref
@pytest.mark.parametrize("B,n,m,k,dup", KNN_CASES)
def test_knn_heap_bit_exact_vs_reference_kernel(B, n, m, k, dup):
    x, q = pc.knn_inputs(B, n, m, k, dup)
    want_idx, want_d2 = ref.knnquery_heap(k, x, q)
    got_idx, got_d2 = fpo.knnquery_heap(k, x, q, return_dist2=True)
    assert torch.equal(got_idx, want_idx)      # including the heap's order of exactly equal distances and the k > n padding
    assert torch.equal(got_d2, want_d2)


@pytest.mark.parametrize("B,n,m,k,dup", KNN_CASES[:5])
def test_knn_heap_matches_cpu_restatement(B, n, m, k, dup):
    x = _cloud(B, n, 3 * n + k, dup)
    q = x[:, torch.randperm(n, generator=torch.Generator().manual_seed(n))[:m]].contiguous()
    assert torch.equal(fpo.knnquery_heap(k, x.to(DEV), q.to(DEV)).cpu(), port_paconv.knnquery_heap(k, x, q))


@needs_ref
@pytest.mark.parametrize("B,n,m,dup", NN_CASES)
def test_three_nn_bit_exact_vs_reference_kernel(B, n, m, dup):
    u, kn = pc.nn_inputs(B, n, m, dup)
    want_d2, want_idx = ref.nearestneighbor(u, kn)
    got_d2, got_idx = fpo.nearestneighbor(u, kn, squared=True)
    assert torch.equal(got_idx, want_idx)
    assert torch.equal(got_d2, want_d2)


@pytest.mark.parametrize("B,n,m,dup", NN_CASES[:3])
def test_three_nn_matches_cpu_restatement(B, n, m, dup):
    u, kn = _cloud(B, n, n + 7 * m), _cloud(B, m, m)
    d, i = port_paconv.nearestneighbor(u, kn)
    gd2, gi = fpo.nearestneighbor(u.to(DEV), kn.to(DEV), squared=True)
    assert torch.equal(gi.cpu(), i) and torch.equal(torch.sqrt(gd2.cpu()), d)    # same sqrt implementation on both sides


@needs_ref
def test_interpolation_and_grouping_vs_reference_kernels():
    feats, idx, w, gidx, fidx = pc.interp_group_gather_inputs(fpo)
    assert torch.equal(fpo.interpolation(feats, idx, w), ref.interpolation(feats, idx, w))
    assert torch.equal(fpo.grouping(feats, gidx), ref.grouping(feats, gidx))
    assert torch.equal(fpo.gathering(feats, fidx), ref.gathering(feats, fidx))


def test_outputs_equal_pinned_digests():
    """Every output of every case above (indices, squared distances, interpolated / grouped / gathered features) is bit-identical
    to this project's pinned outputs.  A regression check of these kernels, not a comparison with the reference."""
    got, want = pc.output_digests(fpo), pc.load_pinned()
    assert sorted(got) == sorted(want)
    assert [k for k in sorted(got) if got[k] != want[k]] == []


@needs_ref
def test_pointops_timing_vs_reference_kernels(capsys):
    """Not an assertion on speed -- prints the device time of each op next to the reference's own kernel compiled for
    sm_100a, at the PAConv embedder's level-0 shapes and 128 clouds (the bench batch).  scripts/pointops_bench.py writes the
    same table to profiles/."""
    from scripts.pointops_bench import table
    rows = table(B=128)
    with capsys.disabled():
        for r in rows:
            print("  ", r)
    assert all(r["match"] for r in rows)
