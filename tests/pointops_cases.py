"""Cases and inputs of the pointops GPU tests (tests/test_pointops_gpu.py), and the pinned outputs of this project's pointops
kernels on them: tests/golden/pointops_pinned.json holds SHA-256 digests (dtype, shape and every byte) of what
flowcompare_b200.pointops returns on every case.

The pins are NOT reference data: they were written by the code they check.  They make any change of these kernels' outputs
visible in a checkout that has no reference tree; agreement with the reference's own kernels is checked only by the
*_vs_reference_kernel tests, which need oracle/_ref/libpointops_ref.so (oracle/build_ref_pointops.sh).  Rewrite the pins only
for a change that is meant to alter these outputs, and run those tests with the reference library when you do.
python -m tests.pointops_cases [out.json]; needs a CUDA device."""
import hashlib
import json
import os
import subprocess
import sys

import torch

PINNED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pointops_pinned.json")
DEV = "cuda:0"

FPS_CASES = [(3, 1250, 312, False), (2, 312, 78, False), (2, 78, 19, False), (2, 19, 4, False), (1, 4096, 1024, False),
             (2, 5000, 1250, False), (2, 1250, 312, True), (1, 2500, 700, True), (1, 33, 33, False)]
KNN_CASES = [(2, 1250, 312, 32, False), (2, 312, 78, 32, False), (2, 78, 19, 32, False), (2, 19, 4, 32, False),
             (2, 1250, 312, 32, True), (1, 700, 700, 16, False), (1, 3000, 129, 40, False)]
NN_CASES = [(2, 1250, 312, False), (2, 312, 78, False), (2, 19, 4, False), (1, 7, 2, False), (2, 1250, 312, True), (1, 5000, 1250, False)]


def cloud(B, n, seed, duplicates=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, n, 3, generator=g) * 2 - 1
    if duplicates:   # the reference's loader oversamples small voxels: exact duplicate points (utils.py:362-370)
        x[:, n // 2:] = x[:, : n - n // 2]
    return x.contiguous()


def digest(t):
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.numpy().tobytes())
    return h.hexdigest()


def key(op, *case):
    return op + ":" + ",".join(str(c) for c in case)


def fps_inputs(B, n, m, dup):
    return cloud(B, n, n + m, dup).to(DEV)


def knn_inputs(B, n, m, k, dup):
    x = cloud(B, n, 3 * n + k, dup).to(DEV)
    return x, x[:, torch.randperm(n, generator=torch.Generator().manual_seed(n))[:m]].contiguous()


def nn_inputs(B, n, m, dup):
    u = cloud(B, n, n + 7 * m, dup).to(DEV)
    return u, (u[:, :m].contiguous() if dup else cloud(B, m, m, False).to(DEV))


def interp_group_gather_inputs(fpo):
    """features [2,67,312], interpolation weights from fpo.nearestneighbor, grouping and gathering indices."""
    g = torch.Generator().manual_seed(3)
    B, c, m, n, k = 2, 67, 312, 1250, 32
    feats = torch.randn(B, c, m, generator=g).to(DEV)
    u, kn = cloud(B, n, 1).to(DEV), cloud(B, m, 2).to(DEV)
    d, idx = fpo.nearestneighbor(u, kn)
    w = 1.0 / (d + 1e-8)
    w = (w / w.sum(dim=2, keepdim=True)).contiguous()
    gidx = torch.randint(0, m, (B, 100, k), generator=g, dtype=torch.int32).to(DEV)
    fidx = torch.randint(0, m, (B, 50), generator=g, dtype=torch.int32).to(DEV)
    return feats, idx, w, gidx, fidx


def output_digests(fpo):
    """key -> {output name: digest} of flowcompare_b200.pointops (`fpo`) on every case."""
    out = {}
    for case in FPS_CASES:
        out[key("fps", *case)] = {"idx": fpo.furthestsampling(fps_inputs(*case), case[2])}
    for case in KNN_CASES:
        x, q = knn_inputs(*case)
        idx, d2 = fpo.knnquery_heap(case[3], x, q, return_dist2=True)
        out[key("knn_heap", *case)] = {"idx": idx, "dist2": d2}
    for case in NN_CASES:
        d2, idx = fpo.nearestneighbor(*nn_inputs(*case), squared=True)
        out[key("three_nn", *case)] = {"dist2": d2, "idx": idx}
    feats, idx, w, gidx, fidx = interp_group_gather_inputs(fpo)
    out["interpolation"] = {"out": fpo.interpolation(feats, idx, w)}
    out["grouping"] = {"out": fpo.grouping(feats, gidx)}
    out["gathering"] = {"out": fpo.gathering(feats, fidx)}
    return {k: {n: digest(t) for n, t in v.items()} for k, v in out.items()}


def load_pinned():
    with open(PINNED) as f:
        return json.load(f)["digests"]


def main():
    from flowcompare_b200 import pointops as fpo
    commit = subprocess.run(["git", "rev-parse", "--short", "HEAD"], capture_output=True, text=True,
                            cwd=os.path.dirname(PINNED)).stdout.strip() or "unknown"
    meta = {"writer": "tests/pointops_cases.py", "source": "flowcompare_b200.pointops (this project's kernels, not the reference)",
            "commit": commit, "device": torch.cuda.get_device_name(0)}
    dst = sys.argv[1] if len(sys.argv) > 1 else PINNED
    with open(dst, "w") as f:
        json.dump({"meta": meta, "digests": output_digests(fpo)}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", dst)


if __name__ == "__main__":
    main()
