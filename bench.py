#!/usr/bin/env python
"""Headline benchmark: cloud-pairs/s for per-point log p(x | context)  (BASELINE.json `metric`).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU

A "step" is one `inner_loop` pass (embed the context cloud, score the target cloud, reference
model_initialization.py:206-228) over one batch of B synthetic cloud pairs per GPU.  Workload = BASELINE.json
configs[1]: "summer-terrain (DGCNN Attention/Perceiver, no extra context)" = architecture `dgcnn_attn`
(content of reference config/swept-energy.yaml, SURVEY.md A.1): Nc=1250 context points, N=1024 target
points, 115 coupling layers, random-init weights of that architecture, synthetic data.

One JSON line is printed by rank 0.  `value` = pairs/s with inputs resident in HBM (CUDA events, max
over ranks); `e2e` = pairs/s through `fc_inner_loop_host` with pinned HOST buffers (H2D of the clouds and
eps, D2H of log_prob inside the timed region); `roofline` = the GEMM class (the dominant kernels) timed
with per-launch CUDA events in one extra instrumented step; `cpu_baseline` = the oracle port on the
host cores on a bounded sample.  Multi-GPU: pairs are sharded across ranks (weak scaling, B per rank),
no collective on the data path (a single all_gather of per-cloud mean log-prob after the timed region).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

METRIC = "cloud-pairs/sec for per-point log p(x|ctx)"
UNIT = "pairs/s"
CLASS_NAMES = ["gemm_fp32_ffma", "gemm_tcgen05_3x", "cross_attention", "knn", "edgeconv_gather_max", "other"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="dgcnn_attn")
    ap.add_argument("--batch", type=int, default=128, help="cloud pairs per step per GPU")
    ap.add_argument("--precision", default=os.environ.get("FC_PRECISION", "auto"), choices=["auto", "fp32", "tf32x3", "fp16x3"])
    ap.add_argument("--cpu-pairs", type=int, default=6, help="pairs in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ncu", action="store_true", help="profiling run: 1 warm-up, timed steps only (not a bench value)")
    ap.add_argument("--no-extras", action="store_true", help="skip per_batch / per_config / sweep / strong-scaling extras")
    ap.add_argument("--extras-budget-s", type=float, default=150.0, help="wall-clock budget of the extras")
    ap.add_argument("--n-context", type=int, default=None)
    ap.add_argument("--n-target", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (loss, log_prob, bpd) as DIR/<name>.npy (float32, at most "
                         "64 MB: a fixed sample of log_prob above that); rank 0 only")
    return ap.parse_args()


DUMP_BYTES = 64 << 20       # cap on everything --dump-outputs writes


def dump_outputs(d, loss, lp, bpd):
    """The arrays a caller of the timed path receives, from its last step.  Inputs and weights are seeded, so two builds run
    with the same arguments can be compared output for output.  log_prob [B, N] is 4*B*N bytes (0.5 MB at the default shape);
    above the cap, log_prob_sample.npy holds a fixed sample of its points (seed 0, ascending flat index b*N + n) and
    log_prob_sample_index.npy those flat indices (float64, exact below 2**53)."""
    os.makedirs(d, exist_ok=True)
    lp = lp.detach().float()
    arrays = {"loss": loss.detach().float(), "bpd": bpd.detach().float()}
    budget = DUMP_BYTES - 4096          # room for the .npy headers and the two scalars
    if 4 * lp.numel() <= budget:
        arrays["log_prob"] = lp
    else:
        idx = torch.randperm(lp.numel(), generator=torch.Generator().manual_seed(0))[:budget // 12].sort().values
        arrays["log_prob_sample"] = lp.reshape(-1)[idx.to(lp.device)]
        arrays["log_prob_sample_index"] = idx.double()
    for name, t in arrays.items():
        np.save(os.path.join(d, name + ".npy"), t.cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline(cfg, pairs, seed=0):
    """Times the oracle port (the reference algorithm restated on CPU, oracle/port.py) on the host cores.
    /root/reference does not exist on the GPU box, so kind is "port"."""
    from flowcompare_b200 import configs, spec
    from oracle import port
    torch.set_num_threads(os.cpu_count())
    fsd, esd = spec.random_state_dicts(cfg, seed=seed)
    dcfg = configs.derive(cfg)
    batch = spec.synthetic_batch(cfg, 1, seed=1)
    args = (batch["extract_0"], batch["extract_1"], batch["extra_context"])
    with torch.no_grad():
        port.inner_loop(args, fsd, esd, dcfg, batch["eps"])  # warm-up
        t0 = time.perf_counter()
        for _ in range(pairs):
            port.inner_loop(args, fsd, esd, dcfg, batch["eps"])
        dt = time.perf_counter() - t0
    return pairs / dt, dt


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host threads, B=1 per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from flowcompare_b200 import configs, spec
    from oracle import port
    cfg = configs.get_config(args.config)
    torch.set_num_threads(os.cpu_count())
    fsd, esd = spec.random_state_dicts(cfg, seed=0)
    dcfg = configs.derive(cfg)
    batch = spec.synthetic_batch(cfg, 1, seed=1, n_context=args.n_context, n_target=args.n_target)
    a = (batch["extract_0"], batch["extract_1"], batch["extra_context"])
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            port.inner_loop(a, fsd, esd, dcfg, batch["eps"])
        t0 = time.perf_counter()
        for _ in range(args.steps):
            loss, lp, bpd = port.inner_loop(a, fsd, esd, dcfg, batch["eps"])
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, loss, lp, bpd)
    v = args.steps / dt
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args, cfg, 1, "cpu"),
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                            "sample": f"{args.steps} steps x 1 pair (Nc={batch['extract_0'].shape[1]}, N={batch['extract_1'].shape[1]}), "
                                      "oracle/port.py = reference algorithm in torch CPU fp32 (reference tree is absent on the GPU box)"},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def workload_config(args, cfg, B, where):
    from flowcompare_b200 import configs
    return {"workload": configs.BASELINE_LABEL.get(args.config, args.config), "architecture": args.config,
            "reference_yaml": configs.REFERENCE_YAML.get(args.config), "pairs_per_step_per_gpu": B,
            "n_context": args.n_context or cfg["n_samples_context"], "n_target": args.n_target or cfg["sample_size"],
            "n_flow_layers": cfg["n_flow_layers"], "latent_dim": cfg["latent_dim"], "sharding": "pairs across ranks",
            "l2": "per-step working set (653 MB weights + >0.5 GB activations) exceeds the 126 MB L2; no explicit flush",
            "where": where}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed `ncu --set full`
    capture (profiles/r02_gemm_tc_ncu_full_summary.csv, made by scripts/ncu_summarize.py).  Static evidence, not
    measured in this run: bench.py never runs under a profiler."""
    path = os.path.join(ROOT, "profiles", "r02_gemm_tc_ncu_full_summary.csv")   # first row: M=65536, N=K=512, GELU
    try:
        import csv
        with open(path) as f:
            row = next(csv.DictReader(f))
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        tot = 0.0
        for k, v in row.items():
            if k.startswith("dram__bytes_read.sum [") or k.startswith("dram__bytes_write.sum ["):
                tot += float(v) * mult[k[k.index("[") + 1:-1]]
        return int(tot), ("ncu --set full, one gemm_tc_kernel launch M=65536 N=512 K=512 GELU (scripts/gemm_one.py): DRAM bytes of "
                          "that launch; its algorithmic bytes are 4*(M*K + M*N) + 4*N*K = 269.5e6 (fp16 hi + lo weights), i.e. no re-reads (L2 keeps "
                          "part of the output)")
    except Exception as exc:  # profile not present
        return None, f"no committed ncu capture readable: {exc}"


def ffma_peak():
    """Measured fp32 FFMA rate of a B200 of this pool in TFLOP/s (profiles/r02_unit_peaks.txt, scripts/micro/peaks.cu; CUDA
    events, no profiler): the denominator of the FMA-bound kernel classes.  None if the file is not readable."""
    try:
        import re
        with open(os.path.join(ROOT, "profiles", "r02_unit_peaks.txt")) as f:
            m = re.search(r"fp32 FFMA\s*:\s*([0-9.]+) TFLOP/s", f.read())
        return float(m.group(1)) if m else None
    except Exception:
        return None


def _timed(fn, steps, warmup=2):
    """pairs-agnostic device timing of fn(): CUDA events on the current stream, after warm-up."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def extras_single_gpu(args, eng, cfg, dev, precision, t_end, note):
    """Extra keys measured on rank 0 at N = 1 after the headline numbers (same engine / weights; device-resident inputs,
    CUDA events).  SURVEY 8d: batch sizes B in {1, 8, 20, 64} of config 2, the other architectures (BASELINE configs[0],
    [2], [3] + PAConv with extra context) at the bench batch, and the point-count sweep of configs[4] on one GPU."""
    from flowcompare_b200 import configs, engine, spec
    out = {}

    def left():
        return t_end - time.perf_counter()

    # ---- batch sizes: eager launches vs one CUDA-graph launch (the forward is ~4.6 k kernel launches)
    per_batch = {}
    for B in (1, 8, 20, 64):
        if left() < 20:
            break
        b = spec.synthetic_batch(cfg, B, seed=7)
        e0, e1, eps = b["extract_0"].to(dev), b["extract_1"].to(dev), b["eps"].to(dev)
        ex = None if b["extra_context"] is None else b["extra_context"].to(dev)
        steps = 4 if B >= 20 else 8
        ms = _timed(lambda: eng.inner_loop((e0, e1, ex), eps=eps), steps)
        rec = {"pairs_per_s": round(B / ms * 1e3, 2), "ms_per_step": round(ms, 3)}
        try:
            run = eng.capture_inner_loop(B, e0.shape[1], e1.shape[1])
            lp_graph = run(e0, e1, ex, eps)[1].clone()
            lp_eager = eng.inner_loop((e0, e1, ex), eps=eps)[1]
            msg = _timed(lambda: run(e0, e1, ex, eps, copy=False), steps)
            rec.update({"cuda_graph_pairs_per_s": round(B / msg * 1e3, 2), "cuda_graph_ms_per_step": round(msg, 3),
                        "cuda_graph_equals_eager": bool(torch.equal(lp_graph, lp_eager))})
            del run
        except Exception as exc:   # keep the bench line alive; the failure is reported
            rec["cuda_graph_error"] = repr(exc)[:200]
        per_batch[str(B)] = rec
    out["per_batch"] = per_batch
    note("extras: per_batch done")

    # ---- the other architectures at the bench batch
    per_config = {}
    for label in ("dgcnn_global", "paconv_attn", "dgcnn_attn_extra", "paconv_attn_extra"):
        if left() < 35:
            per_config[label] = "skipped (extras budget)"
            continue
        c2 = configs.get_config(label)
        fsd, esd = spec.random_state_dicts(c2, seed=0)
        e2 = engine.FlowCompareB200((fsd, esd), c2, device=dev, precision=precision)
        del fsd, esd
        b = spec.synthetic_batch(c2, args.batch, seed=100)
        e0, e1, eps = b["extract_0"].to(dev), b["extract_1"].to(dev), b["eps"].to(dev)
        ex = None if b["extra_context"] is None else b["extra_context"].to(dev)
        ms = _timed(lambda: e2.inner_loop((e0, e1, ex), eps=eps), 3, warmup=2)
        per_config[label] = {"workload": configs.BASELINE_LABEL.get(label, label), "pairs_per_s": round(args.batch / ms * 1e3, 2),
                             "ms_per_step": round(ms, 3), "pairs_per_step": args.batch}
        e2.close()
        del e2, e0, e1, eps
        torch.cuda.empty_cache()
    out["per_config"] = per_config
    note("extras: per_config done")

    # ---- BASELINE configs[4]: point-count sweep Nc = N, same architecture, pairs per step chosen to keep ~131 k target points
    sweep = {}
    for npts in (2048, 4096, 8192, 16384, 32768):
        if left() < 25:
            sweep[str(npts)] = "skipped (extras budget)"
            continue
        B = max(1, min(64, 131072 // npts))
        g = torch.Generator().manual_seed(npts)
        e0 = (torch.rand(B, npts, 6, generator=g) * 2 - 1).to(dev)
        e1 = (torch.rand(B, npts, 6, generator=g) * 2 - 1).to(dev)
        try:
            ms = _timed(lambda: eng.inner_loop((e0, e1, None), eps=None), 2, warmup=1)
            sweep[str(npts)] = {"pairs_per_s": round(B / ms * 1e3, 3), "points_per_s": round(B * npts / ms * 1e3, 1),
                                "ms_per_step": round(ms, 2), "pairs_per_step": B}
        except Exception as exc:
            sweep[str(npts)] = {"error": repr(exc)[:200]}
        del e0, e1
        torch.cuda.empty_cache()
    out["sweep_one_gpu"] = sweep
    note("extras: sweep done")
    return out


def extras_multi_gpu(args, eng, dev, precision, world, rank, note):
    """Extra keys at N > 1 (every rank takes part; times are CUDA-event times, max over ranks, pairs are sharded with no
    data-path collective): BASELINE configs[3] "dulcet-universe (DGCNN Attention + extra context) ... sharded over 2/4/8" at
    SURVEY 8d's 20 pairs per GPU, and configs[4], the point-count sweep Nc = N in {2k..32k} of the bench architecture, with the
    pairs of every point count sharded over the ranks."""
    import torch.distributed as dist
    from flowcompare_b200 import configs, engine, spec
    out = {}

    def timed_all(fn, steps, warmup=1):
        ms = _timed(fn, steps, warmup=warmup)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    c4 = configs.get_config("dgcnn_attn_extra")
    fsd, esd = spec.random_state_dicts(c4, seed=0)
    e4 = engine.FlowCompareB200((fsd, esd), c4, device=dev, precision=precision)
    del fsd, esd
    for B4 in (20, args.batch):
        b = spec.synthetic_batch(c4, B4, seed=200 + rank)
        e0, e1, eps, ex = b["extract_0"].to(dev), b["extract_1"].to(dev), b["eps"].to(dev), b["extra_context"].to(dev)
        ms = timed_all(lambda: e4.inner_loop((e0, e1, ex), eps=eps), 3, warmup=2)
        out[f"pairs_per_gpu_{B4}"] = {"pairs_per_s": round(world * B4 / ms * 1e3, 2), "ms_per_step": round(ms, 3)}
    e4.close()
    del e4
    torch.cuda.empty_cache()
    note("extras: config 4 sharded done")
    sweep = {}
    for npts in (2048, 4096, 8192, 16384, 32768):
        B = max(1, min(64, 131072 // npts))
        g = torch.Generator().manual_seed(npts * 31 + rank)
        e0 = (torch.rand(B, npts, 6, generator=g) * 2 - 1).to(dev)
        e1 = (torch.rand(B, npts, 6, generator=g) * 2 - 1).to(dev)
        ms = timed_all(lambda: eng.inner_loop((e0, e1, None), eps=None), 2, warmup=1)
        sweep[str(npts)] = {"pairs_per_s": round(world * B / ms * 1e3, 3), "points_per_s": round(world * B * npts / ms * 1e3, 1),
                            "ms_per_step": round(ms, 2), "pairs_per_step_per_gpu": B}
        del e0, e1
        torch.cuda.empty_cache()
    note("extras: sharded sweep done")
    return {"config4_dgcnn_attn_extra_sharded": dict(out, workload=configs.BASELINE_LABEL["dgcnn_attn_extra"], ranks=world),
            "sweep_sharded": dict(sweep, ranks=world, workload="point-count sweep, Nc = N, dgcnn_attn")}


def strong_scaling(eng, cfg, dev, world, rank, B_chunk, total_pairs=1024):
    """A FIXED evaluation set of 1024 pairs sharded over the ranks through flowcompare_b200.sharding.evaluate_sharded (the
    host logic of test_flow.evaluate_on_test: score, reduce to the running nats) with the real engine and NCCL: the one
    collective is the gather of per-cloud scalars.  eps is drawn on the device.  Returns pairs/s (max over ranks)."""
    import torch.distributed as dist
    from flowcompare_b200 import sharding
    Nc, N = cfg["n_samples_context"], cfg["sample_size"]
    lo, hi = sharding.shard_bounds(total_pairs, rank, world)
    g = torch.Generator().manual_seed(1234)      # every rank builds the same set and scores its own block
    e0 = torch.rand(total_pairs, Nc, 6, generator=g)
    e1 = torch.rand(total_pairs, N, 6, generator=g)
    e0, e1 = (e0 * 2 - 1).to(dev), (e1 * 2 - 1).to(dev)
    eps_dummy = torch.empty(total_pairs, 0)

    def score(batch, _eps):
        a, b_, _ = batch
        outs = []
        for i in range(0, a.shape[0], B_chunk):
            outs.append(eng.inner_loop((a[i:i + B_chunk], b_[i:i + B_chunk], None), eps=None)[1])
        return torch.cat(outs)

    sharding.evaluate_sharded(score, e0[: 2 * world], e1[: 2 * world], None, eps_dummy[: 2 * world])   # warm-up incl. the collective
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    per_cloud, nats = sharding.evaluate_sharded(score, e0, e1, None, eps_dummy)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"pairs": total_pairs, "pairs_per_s": round(total_pairs / t.item(), 2), "seconds": round(t.item(), 3), "nats": nats,
            "ranks": world, "collective": "one all_gather of per-cloud mean log-prob (NCCL)" if world > 1 else "none",
            "local_pairs": hi - lo}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    t_start = time.perf_counter()

    def note(what):   # phase trace on stderr (stdout carries exactly one JSON line)
        print(f"[bench rank {os.environ.get('RANK', '0')}] {time.perf_counter() - t_start:7.1f}s {what}", file=sys.stderr, flush=True)

    from flowcompare_b200 import configs, engine, lib, spec
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch.distributed as dist
    # stdout carries exactly one JSON line: keep NCCL's banner ("NCCL version ...", printed at NCCL_DEBUG=VERSION) off it
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    note("process group ready" if world > 1 else "start")
    torch.set_grad_enabled(False)

    cfg = configs.get_config(args.config)
    if args.n_target:
        cfg["sample_size"] = args.n_target
    B = args.batch
    precision = args.precision
    clib = lib.load()
    if precision == "auto":
        precision = "fp16x3"   # tensor-core path (3xFP16 error-compensated); parity-tested at full depth like the exact-fp32 FFMA path
    fsd, esd = spec.random_state_dicts(cfg, seed=0)          # same weights on every rank
    eng = engine.FlowCompareB200((fsd, esd), cfg, device=dev, precision=precision)
    del fsd, esd
    note("weights packed and uploaded")
    batch = spec.synthetic_batch(cfg, B, seed=100 + rank, n_context=args.n_context, n_target=args.n_target)
    Nc, N = batch["extract_0"].shape[1], batch["extract_1"].shape[1]
    e0, e1, eps = batch["extract_0"].to(dev), batch["extract_1"].to(dev), batch["eps"].to(dev)
    extra = None if batch["extra_context"] is None else batch["extra_context"].to(dev)
    gathered = [torch.empty(B, device=dev) for _ in range(world)] if world > 1 else None

    def step():   # rank-local: pairs are sharded across ranks and nothing is exchanged on the data path
        return eng.inner_loop((e0, e1, extra), eps=eps)

    for _ in range(1 if args.ncu else max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    note("warm-up done")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.launch_count()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        loss, lp, bpd = step()
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    note("timed region done")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, lp, bpd)
    if world > 1:   # outside the timed region: collect the per-cloud nats of every rank (what a caller would do once)
        dist.all_gather(gathered, lp.mean(dim=1))
    launches = lib.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    value = world * B * args.steps / (ms / 1e3)
    if args.ncu:
        if rank == 0:
            print(json.dumps({"ncu_run": True, "not_a_bench_value": round(value, 2), "gpu_launches": int(launches)}), flush=True)
        return

    # ---- end to end through the C ABI with host buffers
    pin = lambda x: x.contiguous().pin_memory()
    h0, h1, heps = pin(batch["extract_0"]), pin(batch["extract_1"]), pin(batch["eps"])
    hex_ = None if batch["extra_context"] is None else pin(batch["extra_context"].reshape(-1))
    hlp, hst = torch.empty(B, N).pin_memory(), torch.empty(2).pin_memory()
    for _ in range(2):
        eng.inner_loop_host(h0, h1, hex_, heps, hlp, hst)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.inner_loop_host(h0, h1, hex_, heps, hlp, hst)   # synchronous: returns after the D2H copy
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / t.item()
    h2d = 4 * (h0.numel() + h1.numel() + heps.numel() + (0 if hex_ is None else hex_.numel()))
    d2h = 4 * (hlp.numel() + 2)
    # e2e result must equal the device-resident result
    same = bool(torch.equal(hlp, lp.cpu()))
    # second end-to-end figure: the augmentation noise drawn ON THE DEVICE (fc_fill_normal), so only the clouds cross PCIe
    def e2e_device_eps():
        d0, d1 = h0.to(dev, non_blocking=True), h1.to(dev, non_blocking=True)
        dx = None if hex_ is None else hex_.to(dev, non_blocking=True)
        _, lpd, _ = eng.inner_loop((d0, d1, dx), eps=None)
        hlp.copy_(lpd, non_blocking=True)
        torch.cuda.synchronize()
    for _ in range(2):
        e2e_device_eps()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_device_eps()
    t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_dev_eps_value = world * B * args.steps / t.item()
    h2d_dev_eps = 4 * (h0.numel() + h1.numel() + (0 if hex_ is None else hex_.numel()))

    # ---- one instrumented step: per-class kernel time with CUDA events around every launch
    roofline, classes = None, None
    if rank == 0:
        clib.fc_profile_begin()
        eng.inner_loop((e0, e1, extra), eps=eps)   # rank-local: NO collective here (only rank 0 runs this)
        ms_c = (ctypes.c_double * 6)(); fl_c = (ctypes.c_double * 6)(); by_c = (ctypes.c_double * 6)()
        ln_c = (ctypes.c_int64 * 6)()
        clib.fc_profile_end(ms_c, fl_c, by_c, ln_c, 6)
        total_ms = sum(ms_c)
        classes = {}
        for i, nm in enumerate(CLASS_NAMES):
            if ln_c[i]:
                classes[nm] = {"launches": int(ln_c[i]), "ms": round(ms_c[i], 3), "share": round(ms_c[i] / total_ms, 4),
                               "tflops": round(fl_c[i] / ms_c[i] / 1e9, 2), "gbs": round(by_c[i] / ms_c[i] / 1e6, 1)}
        fpk = ffma_peak()
        for nm in ("knn", "gemm_fp32_ffma"):      # FMA-bound classes against the measured FFMA rate (profiles/r02_unit_peaks.txt)
            if fpk and nm in classes:
                classes[nm]["frac_of_measured_ffma_peak"] = round(classes[nm]["tflops"] / fpk, 4)
        pk = peaks()
        top = 1 if ln_c[1] and ms_c[1] >= ms_c[0] else 0
        achieved = fl_c[top] / ms_c[top] / 1e9
        traffic, traffic_note = ncu_traffic()
        f16 = precision == "fp16x3"
        # what the tensor cores execute: 3 products per algorithmic one; 3xFP16 runs at the bf16/fp16 rate, 3xTF32 at half of it
        issued = 3 * achieved
        issue_peak = pk["bf16_sustained"] if f16 else pk["bf16_sustained"] / 2
        roofline = {"kernel": CLASS_NAMES[top] + ("(fp16)" if f16 else "(tf32)") if top == 1 else CLASS_NAMES[top], "bound": "tensor",
                    "achieved": round(achieved, 2), "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": round(achieved / pk["bf16_sustained"], 4),
                    "traffic": traffic if top == 1 else None, "traffic_note": traffic_note, "peak_source": pk["source"] + ", dense bf16 sustained",
                    "note": "achieved = algorithmic 2*M*N*K flops of every launch of the class / summed CUDA-event time in one "
                            "instrumented step; an fp32-faithful GEMM issues 3 tensor products per algorithmic one, so its ceiling is "
                            + ("1/3 of this peak (3xFP16)" if f16 else "1/6 of this peak (3xTF32: half rate, 3 products)"),
                    "avg_launch_ms": round(ms_c[top] / max(1, ln_c[top]), 4),
                    "issued_tensor_tflops": round(issued, 1) if top == 1 else None,
                    "frac_of_issue_rate_peak": round(issued / issue_peak, 4) if top == 1 else None}

    note("e2e + instrumented step done")
    # live precision evidence: the timed path (3xTF32 on the tensor cores) against the exact-fp32 FFMA path of the same
    # library on 2 pairs of this step's batch (both are parity-tested at full depth against the reference's goldens)
    precision_check = None
    if rank == 0 and precision != "fp32" and not args.ncu:
        fsd, esd = spec.random_state_dicts(cfg, seed=0)
        eng32 = engine.FlowCompareB200((fsd, esd), cfg, device=dev, precision="fp32")
        del fsd, esd
        sub = (e0[:2], e1[:2], None if extra is None else extra[:2])
        lp_tc = eng.inner_loop(sub, eps=eps[:2])[1]
        lp_32 = eng32.inner_loop(sub, eps=eps[:2])[1]
        d = (lp_tc - lp_32).abs()
        precision_check = {"pairs": 2, "max_abs_diff_nats": float(d.max().item()), "median_abs_diff_nats": float(d.median().item()),
                           "mean_rel_diff": float(abs(lp_tc.mean().item() - lp_32.mean().item()) / abs(lp_32.mean().item())),
                           "note": precision + " (timed) vs exact-fp32 FFMA path, 115 layers; the reference's own fp32-vs-fp64 noise at "
                                   "this depth is 2e-3 max / 2.4e-4 mean nats (DESIGN.md section 2)"}
        eng32.close()
        del eng32
        note("precision check done")
    extras = {}
    if not args.no_extras and not args.ncu:
        if world == 1:
            extras = extras_single_gpu(args, eng, cfg, dev, precision, time.perf_counter() + args.extras_budget_s, note)
        else:
            extras = extras_multi_gpu(args, eng, dev, precision, world, rank, note)
        try:
            extras["strong_scaling_fixed_set"] = strong_scaling(eng, cfg, dev, world, rank, B)
        except Exception as exc:
            extras["strong_scaling_fixed_set"] = {"error": repr(exc)[:200]}
        note("extras: strong scaling done")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:   # the CPU baseline is measured at N=1 only
        v, dt = cpu_baseline(cfg, args.cpu_pairs)
        cpu = {"value": round(v, 4), "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
               "sample": f"{args.cpu_pairs} pairs (B=1 per call, Nc=1250, N=1024, same architecture and weights), {dt:.1f} s of "
                         "oracle/port.py (reference algorithm, torch CPU fp32, all host threads)"}

    if rank == 0:
        out = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f32" if precision == "fp32" else precision + "(f32-faithful)",
               "data": "synthetic", "config": workload_config(args, cfg, B, "B200"),
               "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "matches_device_resident_result": same,
                       "device_drawn_eps": {"value": round(e2e_dev_eps_value, 3), "unit": UNIT, "h2d_bytes_per_step": h2d_dev_eps,
                                            "d2h_bytes_per_step": 4 * hlp.numel(),
                                            "note": "same call path through engine.inner_loop with host clouds; the noise is drawn by fc_fill_normal on the device"}},
               "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernel_classes": classes,
               "cpu_baseline": cpu, "mean_log_prob": float(lp.mean().item()), "bpd": float(bpd.item()),
               "precision_check": precision_check, "weights_mb": round(eng.weight_bytes() / 1e6, 1)}
        out.update(extras)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()                 # every rank leaves together (rank 0 did the rank-local extras above)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
