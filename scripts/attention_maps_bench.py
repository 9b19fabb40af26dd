"""Cost of the attention maps (csrc/attention_maps.cu, engine.attention_maps).

1. attention_maps_kernel alone (fc_attention_maps, CUDA events around many back-to-back launches) at the bench shape
   (128 clouds x 1024 queries x 1250 keys) and at 4 clouds x 8192 x 8192: achieved FFMA rate against the measured fp32 FFMA
   peak (profiles/r02_unit_peaks.txt), HBM write rate against the data sheet, and which of the two bounds the kernel.
   The outputs (655 MB, 1.07 GB) are larger than the 126 MB L2, so the writes reach HBM; q and k (<= 100 MB) stay in L2.
2. A 128-pair forward of the full-depth DGCNN-attention model (3xFP16) with no block, one block and 8 blocks captured.

Prints the card's name and power limit first: the numbers belong to them.  Usage: python scripts/attention_maps_bench.py
"""
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


def kernel(lib, B, N, Nc, launches):
    g = torch.Generator(device=DEV).manual_seed(B + N + Nc)
    q = torch.randn(B * N, 64, device=DEV, generator=g) * 0.5
    kv = torch.randn(B * Nc, 128, device=DEV, generator=g)
    out = torch.empty(B, N, Nc, device=DEV)
    st = torch.cuda.current_stream().cuda_stream

    def call():
        assert lib.fc_attention_maps(q.data_ptr(), 64, kv.data_ptr(), 128, 0, N, out.data_ptr(), B, N, Nc, 0.125, st) == 0

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    # the first rows of cloud 0 against fp64
    want = torch.softmax((q[:8].double() @ kv[:Nc, :64].double().t()) * 0.125, dim=-1)
    err = (out[0, :8].double() - want).abs().max().item()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    elems = B * N * Nc
    flop = 256.0 * elems                         # two passes of a 64-long fma chain per weight
    wbytes = 4.0 * elems
    rate, bw = flop / (ms * 1e-3), wbytes / (ms * 1e-3)
    t_ffma, t_hbm = flop / FFMA_PEAK, wbytes / HBM_PEAK
    bound = "FFMA" if t_ffma >= t_hbm else "HBM writes"
    print(f"kernel B={B} N={N} Nc={Nc}: {ms:.3f} ms per launch ({launches} launches), {rate / 1e12:.1f} TFLOP/s = "
          f"{rate / FFMA_PEAK:.2f} of the FFMA peak, {bw / 1e12:.2f} TB/s written = {bw / HBM_PEAK:.2f} of HBM; "
          f"bound: {bound} (lower bounds {t_ffma * 1e3:.3f} ms FFMA, {t_hbm * 1e3:.3f} ms HBM: "
          f"{max(t_ffma, t_hbm) * 1e3 / ms:.2f} of it reached); max |P - fp64| {err:.2e}", flush=True)


def forward(B=128, rounds=5):
    cfg = configs.get_config("dgcnn_attn")
    fsd, esd = spec.random_state_dicts(cfg, seed=0)
    batch = spec.synthetic_batch(cfg, B, seed=100)
    e = eng.FlowCompareB200((fsd, esd), cfg, device=DEV, precision="fp16x3")
    ctx = e.embed(batch["extract_0"].to(DEV))
    x, eps = batch["extract_1"].to(DEV), batch["eps"].to(DEV)
    names = e.attention_layer_names
    variants = {
        "no block (log_prob)": lambda: e.log_prob(x, ctx, eps=eps),
        "1 block": lambda: e.attention_maps(x, ctx, eps=eps, layers=[names[58]]),
        "8 blocks": lambda: e.attention_maps(x, ctx, eps=eps, layers=names[::15][:8]),
    }
    for f in variants.values():
        for _ in range(2):
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):                      # interleaved, so drift of the clocks hits every variant alike
        for k, f in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
            del r
    base = sorted(times["no block (log_prob)"])[rounds // 2]
    for k, ts in times.items():
        ts = sorted(ts)
        med = ts[rounds // 2]
        print(f"forward B={B} (115 layers, fp16x3), {k}: median {med:.2f} ms (min {ts[0]:.2f}, max {ts[-1]:.2f}), "
              f"+{med - base:.2f} ms over the plain forward", flush=True)
    e.close()


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.set_grad_enabled(False)
    print("card (name, power limit, max SM clock, SM clock):", card(), flush=True)
    lib = fclib.load()
    kernel(lib, 128, 1024, 1250, 50)
    kernel(lib, 4, 8192, 8192, 20)
    forward()
    print("card after the run:", card(), flush=True)


if __name__ == "__main__":
    main()
