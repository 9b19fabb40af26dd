"""Cost of the attention score gradients (csrc/attention_score_grad.cu, engine.attention_score_grads).

1. attention_score_grad_kernel alone (fc_attention_score_grad, CUDA events around many back-to-back launches) at the bench shape,
   64 clouds x 1024 queries x 1250 keys, storing and accumulating: achieved FFMA rate against the measured fp32 FFMA peak
   (profiles/r02_unit_peaks.txt), HBM traffic against the data sheet, and which of the two bounds the kernel.  The output
   (328 MB) is larger than the 126 MB L2, so its writes reach HBM; q, k|v, o and dO (< 100 MB) stay in L2.
2. attention_score_grads against log_prob_grad on the bench configuration (DGCNN-attention, 115 layers, 3xFP16, 1024 points
   against a 1250-point context) at B = 8, 32, 64: one block, all 116 blocks summed (sum_layers) and, at B = 8 only, all 116
   blocks written separately (4.9 GB).  Medians of CUDA-event times over `--rounds` interleaved calls after one warm-up call each.

Prints the card's name and power limit first and last (the numbers belong to them) and one JSON line at the end.
Usage: python scripts/attention_score_grads_bench.py [--rounds 3] [--batches 8,32,64]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from flowcompare_b200 import configs, engine as eng, lib as fclib, spec  # noqa: E402

FFMA_PEAK = 72.5e12     # measured fp32 FFMA rate of a B200 (profiles/r02_unit_peaks.txt)
HBM_PEAK = 7.7e12       # data sheet, one B200
DEV = "cuda:0"


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        return f"nvidia-smi not available ({ex}); torch: {torch.cuda.get_device_name(0)}"


def kernel(lib, B, N, Nc, launches, accumulate):
    g = torch.Generator(device=DEV).manual_seed(B + N + Nc)
    q = torch.randn(B * N, 64, device=DEV, generator=g) * 0.5
    kv = torch.randn(B * Nc, 128, device=DEV, generator=g)
    dO = torch.randn(B * N, 64, device=DEV, generator=g)
    P = torch.softmax((q.view(B, N, 64) @ kv.view(B, Nc, 128)[..., :64].transpose(1, 2)) * 0.125, dim=-1)
    o = (P @ kv.view(B, Nc, 128)[..., 64:]).reshape(B * N, 64).contiguous()
    del P
    out = torch.zeros(B, N, Nc, device=DEV)
    st = torch.cuda.current_stream().cuda_stream

    def call():
        assert lib.fc_attention_score_grad(q.data_ptr(), 64, kv.data_ptr(), 128, o.data_ptr(), 64, dO.data_ptr(), 64, 0, N,
                                           out.data_ptr(), accumulate, B, N, Nc, 0.125, st) == 0

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    elems = B * N * Nc
    flop = 384.0 * elems                         # a 64-long fma chain in pass 1, two in pass 2
    hbm = (8.0 if accumulate else 4.0) * elems   # written (and, accumulating, read back)
    rate, bw = flop / (ms * 1e-3), hbm / (ms * 1e-3)
    t_ffma, t_hbm = flop / FFMA_PEAK, hbm / HBM_PEAK
    bound = "FFMA" if t_ffma >= t_hbm else "HBM"
    mode = "accumulate" if accumulate else "store"
    print(f"kernel ({mode}) B={B} N={N} Nc={Nc}: {ms:.3f} ms per launch ({launches} launches), {rate / 1e12:.1f} TFLOP/s = "
          f"{rate / FFMA_PEAK:.2f} of the FFMA peak, {bw / 1e12:.2f} TB/s of output traffic = {bw / HBM_PEAK:.2f} of HBM; "
          f"bound: {bound} (lower bounds {t_ffma * 1e3:.3f} ms FFMA, {t_hbm * 1e3:.3f} ms HBM: "
          f"{max(t_ffma, t_hbm) * 1e3 / ms:.2f} of it reached)", flush=True)
    return {"mode": mode, "B": B, "N": N, "Nc": Nc, "ms": ms, "tflops": rate / 1e12, "of_ffma_peak": rate / FFMA_PEAK}


def timed(f):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = f()
    e1.record()
    torch.cuda.synchronize()
    del r
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batches", default="8,32,64")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.set_grad_enabled(False)
    c = card()
    print("card (name, power limit, max SM clock, SM clock):", c, flush=True)
    lib = fclib.load()
    res = {"card": c, "config": "dgcnn_attn, 115 layers, fp16x3, N=1024, Nc=1250", "kernel": [], "runs": []}
    for acc in (0, 1):
        res["kernel"].append(kernel(lib, 64, 1024, 1250, 30, acc))
    torch.cuda.empty_cache()
    cfg = configs.get_config("dgcnn_attn")
    fsd, esd = spec.random_state_dicts(cfg, seed=0)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    names = e.attention_layer_names
    for B in [int(b) for b in args.batches.split(",")]:
        batch = spec.synthetic_batch(cfg, B, seed=100)
        ctx = e.embed(batch["extract_0"].to(DEV))
        x = batch["extract_1"].to(DEV)
        eps = e.draw_eps(B, x.shape[1], seed=5)
        variants = {
            "log_prob_grad": lambda: e.log_prob_grad(x, ctx, eps=eps),
            "1 block": lambda: e.attention_score_grads(x, ctx, eps=eps, layers=[names[58]]),
            "116 blocks summed": lambda: e.attention_score_grads(x, ctx, eps=eps, sum_layers=True),
        }
        if B == 8:
            variants["116 blocks separate"] = lambda: e.attention_score_grads(x, ctx, eps=eps)
        for f in variants.values():
            timed(f)
        times = {k: [] for k in variants}
        for _ in range(args.rounds):             # interleaved, so drift of the clocks hits every variant alike
            for k, f in variants.items():
                times[k].append(timed(f))
        run = {"B": B}
        base = sorted(times["log_prob_grad"])[args.rounds // 2]
        for k, ts in times.items():
            ts = sorted(ts)
            ms = ts[args.rounds // 2]
            run[k] = {"ms": ms, "pairs_per_s": B / (ms * 1e-3), "over_log_prob_grad_ms": ms - base}
            print(f"B={B:3d} {k:20s}: median {ms:9.1f} ms (min {ts[0]:.1f}, max {ts[-1]:.1f}), {B / (ms * 1e-3):7.1f} pairs/s, "
                  f"+{ms - base:.1f} ms over log_prob_grad", flush=True)
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
