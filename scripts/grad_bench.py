"""Cost of the input gradients (engine.log_prob_grad) against the forward pass (engine.log_prob) on the bench configuration:
DGCNN-attention, 115 flow layers, 3xFP16, 1024 points scored against a 1250-point context, at B = 8, 32 and 64 cloud pairs.

Pairs per second are medians of CUDA-event times over `--rounds` interleaved calls after one warm-up call each (each call ends in
a device synchronise).  The per-phase split of one gradient call comes from the library's per-class event profiler: the
checkpointing forward is timed as `log_prob`'s profiled kernels, the recompute as one more forward, the transposed GEMMs as the
gradient call's GEMM time minus twice the forward's, the dQ kernel as its attention time minus twice the forward's; the rest of the
call's wall time (elementwise kernels, checkpoint copies, launch gaps) is reported as "other".
Prints the card's name and power limit first (the times belong to them) and one JSON line at the end.
Usage: python scripts/grad_bench.py [--rounds 3] [--batches 8,32,64]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from flowcompare_b200 import configs, engine as eng, spec  # noqa: E402

DEV = "cuda:0"
CLASSES = ["gemm_ffma", "gemm_tc", "attention", "knn", "edgeconv", "other"]


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        return f"nvidia-smi not available ({ex}); torch: {torch.cuda.get_device_name(0)}"


def timed(f):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def profiled(lib, f):
    """ms per kernel class of one call (the library's event profiler)."""
    n = len(CLASSES)
    ms, fl, by, la = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_int64 * n)()
    torch.cuda.synchronize()
    lib.fc_profile_begin()
    f()
    torch.cuda.synchronize()
    lib.fc_profile_end(ms, fl, by, la, n)
    return dict(zip(CLASSES, list(ms)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batches", default="8,32,64")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.set_grad_enabled(False)
    c = card()
    print("card (name, power limit, max SM clock, SM clock):", c, flush=True)
    cfg = configs.get_config("dgcnn_attn")
    fsd, esd = spec.random_state_dicts(cfg, seed=0)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    res = {"card": c, "config": "dgcnn_attn, 115 layers, fp16x3, N=1024, Nc=1250", "runs": []}
    for B in [int(b) for b in args.batches.split(",")]:
        batch = spec.synthetic_batch(cfg, B, seed=100)
        ctx = e.embed(batch["extract_0"].to(DEV))
        x = batch["extract_1"].to(DEV)
        eps = e.draw_eps(B, x.shape[1], seed=5)
        variants = {"log_prob": lambda: e.log_prob(x, ctx, eps=eps), "log_prob_grad": lambda: e.log_prob_grad(x, ctx, eps=eps)}
        for f in variants.values():
            f()
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(args.rounds):
            for k, f in variants.items():
                times[k].append(timed(f))
        run = {"B": B}
        for k, ts in times.items():
            ms = sorted(ts)[len(ts) // 2]
            run[k] = {"ms": ms, "pairs_per_s": B / (ms * 1e-3)}
            print(f"B={B:3d} {k:13s}: median {ms:9.1f} ms (min {min(ts):.1f}, max {max(ts):.1f}), {B / (ms * 1e-3):7.1f} pairs/s",
                  flush=True)
        pf, pg = profiled(e.lib, variants["log_prob"]), profiled(e.lib, variants["log_prob_grad"])
        gemm_f, gemm_g = pf["gemm_ffma"] + pf["gemm_tc"], pg["gemm_ffma"] + pg["gemm_tc"]
        phases = {"checkpointing forward": sum(pf.values()), "recompute": sum(pf.values()),
                  "transposed GEMMs": gemm_g - 2 * gemm_f, "dQ": pg["attention"] - 2 * pf["attention"]}
        # the elementwise kernels and the checkpoint copies are not in the profiler's classes: the rest of the wall time
        phases["other (elementwise kernels, copies, gaps)"] = run["log_prob_grad"]["ms"] - sum(pg.values())
        run["phases_ms"] = phases
        print(f"B={B:3d} phases (profiled kernel time, ms): " + ", ".join(f"{k} {v:.1f}" for k, v in phases.items()), flush=True)
        res["runs"].append(run)
        del ctx, x, eps
        e._ws = None
        torch.cuda.empty_cache()
    res["card_after"] = card()
    print("card after the run:", res["card_after"], flush=True)
    print(json.dumps(res), flush=True)
    e.close()


if __name__ == "__main__":
    main()
