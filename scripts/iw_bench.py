"""Cost and effect of the multi-draw log-likelihood (engine.log_prob_iw).

1. Time: `log_prob_iw` at K in {1, 4, 16} draws on the bench configuration (DGCNN-attention, 115 flow layers, 3xFP16, 1024
   points scored against a 1250-point context, B = 32 and 128 cloud pairs), against K separate `log_prob` calls on the same
   embedding, as draws x pairs per second.  Each variant runs once to warm up, then `--rounds` times interleaved with the
   others; medians of CUDA-event times (each call ends in a device synchronise).
2. Noise: over 8 seeds of the draws, the median per-point standard deviation of the estimate and the fraction of points whose
   change mask (log_prob_to_change, multiple = 3) differs between two seeds, as functions of K.  The weights are seeded
   `spec.random_state_dicts`, not a trained checkpoint: these numbers show how the estimator behaves, not what a trained
   model gains.

Prints the card's name and power limit first (the times belong to them) and one JSON line at the end.
Usage: python scripts/iw_bench.py [--rounds 3] [--noise-pairs 16]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from flowcompare_b200 import configs, engine as eng, spec  # noqa: E402

DEV = "cuda:0"


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


def time_section(e, cfg, rounds):
    out = []
    for B in (32, 128):
        batch = spec.synthetic_batch(cfg, B, seed=100)
        ctx = e.embed(batch["extract_0"].to(DEV))
        x = batch["extract_1"].to(DEV)
        variants = {}
        for K in (1, 4, 16):
            variants[("log_prob_iw", K)] = lambda K=K: e.log_prob_iw(x, ctx, n_draws=K)
            variants[("K x log_prob", K)] = lambda K=K: [e.log_prob(x, ctx) for _ in range(K)]
        for f in variants.values():
            f()
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(rounds):
            for k, f in variants.items():
                times[k].append(timed(f))
        for (what, K), ts in times.items():
            ms = sorted(ts)[len(ts) // 2]
            rate = K * B / (ms * 1e-3)
            print(f"B={B} K={K:2d} {what:13s}: median {ms:9.1f} ms (min {min(ts):.1f}, max {max(ts):.1f}), "
                  f"{rate:7.1f} draws*pairs/s", flush=True)
            out.append({"B": B, "K": K, "variant": what, "ms": ms, "draws_pairs_per_s": rate})
        del ctx, x
        torch.cuda.empty_cache()
    return out


def noise_section(e, cfg, pairs, seeds=8, Ks=(1, 2, 4, 8, 16)):
    """lp_1|0: the N target points given context cloud 0; lp_0|0: N points of cloud 0 itself given the same context."""
    batch = spec.synthetic_batch(cfg, pairs, seed=300)
    N = batch["extract_1"].shape[1]
    ctx = e.embed(batch["extract_0"].to(DEV))
    x = torch.cat([batch["extract_1"], batch["extract_0"][:, :N]]).to(DEV)
    ctx2 = torch.cat([ctx, ctx])
    out = []
    for K in Ks:
        est = []
        for s in range(seeds):
            g = torch.Generator(device=DEV).manual_seed(1000 * s + K)
            eps = torch.randn(K, 2 * pairs, N, e.D - e.d_in, device=DEV, generator=g)
            est.append(e.log_prob_iw(x, ctx2, n_draws=K, eps=eps))
            del eps
        est = torch.stack(est)                                                  # [seeds, 2*pairs, N]
        std = est.double().std(dim=0).median().item()
        masks = [eng.log_prob_to_change(v[:pairs], v[pairs:], 3.0) > 0 for v in est]
        flips = sum((masks[i] != masks[i + 1]).double().mean().item() for i in range(0, seeds, 2)) / (seeds // 2)
        changed = sum(m.double().mean().item() for m in masks) / seeds
        print(f"K={K:2d}: median per-point std over {seeds} seeds {std:8.3f} nats; change mask (multiple=3) differs between "
              f"two seeds on {flips * 100:6.2f} % of points ({changed * 100:.2f} % marked changed on average)", flush=True)
        out.append({"K": K, "median_point_std_nats": std, "mask_flip_fraction": flips, "changed_fraction": changed})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--noise-pairs", type=int, default=16)
    ap.add_argument("--skip-time", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.set_grad_enabled(False)
    c = card()
    print("card (name, power limit, max SM clock, SM clock):", c, flush=True)
    cfg = configs.get_config("dgcnn_attn")
    fsd, esd = spec.random_state_dicts(cfg, seed=0)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    res = {"card": c, "config": "dgcnn_attn, 115 layers, fp16x3, N=1024, Nc=1250, untrained seeded weights"}
    if not args.skip_time:
        res["time"] = time_section(e, cfg, args.rounds)
    res["noise"] = noise_section(e, cfg, args.noise_pairs)
    res["card_after"] = card()
    print("card after the run:", res["card_after"], flush=True)
    print(json.dumps(res), flush=True)
    e.close()


if __name__ == "__main__":
    main()
