#!/usr/bin/env python
"""bench.py - headline benchmark of the UniVTG hot path on B200 (contract in the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic batch:
  cfg3_train BASELINE.json configs[2]: B=32, L_v=75, L_t=32, d=1024, 4 layers: forward + criterion + backward + grad-clip +
             AdamW - the metric BASELINE.json quotes ("pairs/sec (fwd+bwd)")                               [default]
  cfg2_fwd   configs[1]: same shapes, inference forward (also reported as "forward_only" inside the default line)
  cfg4_train configs[3]: per-rank shard of the vlp_ddp batch (B=32/rank, L_v=150); cfg4_fwd / cfg5_fwd: forward only
Metric: video-query pairs/sec (whole job, all ranks).  `value` is measured with inputs resident in HBM; `e2e` through the
public plugin API (`model(**inputs)`) with pinned HOST inputs, H2D + D2H inside the timed region.
N>1: one process per GPU (torchrun), each rank runs its own replica on its own batch (the path shards by sample; inference
needs no collective) -> "scaling": "weak".
--impl reference: the CPU arm (the oracle port of the reference's fp32 PyTorch path, all host threads), rank 0 only.
--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step computed to DIR/<name>.npy (see dump_outputs).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from univtg_b200 import synth  # noqa: E402

WORKLOADS = {
    "cfg2_fwd": dict(cfg="cfg2", mode="fwd"),
    "cfg4_fwd": dict(cfg="cfg4", mode="fwd"),
    "cfg5_fwd": dict(cfg="cfg5", mode="fwd"),
    # BASELINE.json configs[2]: cfg2 shapes, criterion (5 losses) + backward + grad-clip + AdamW (train_vlp_ddp.py:56-68)
    "cfg3_train": dict(cfg="cfg2", mode="train"),
    # configs[3]: per-rank shard (B=32, L_v=150) of the vlp_ddp pre-training batch; N ranks -> global batch 32 N
    "cfg4_train": dict(cfg="cfg4", mode="train"),
}
# BASELINE.json's metric is "video-query pairs/sec (fwd+bwd) at L_v=75, d=1024": the full train step on cfg2 shapes.
DEFAULT_WORKLOAD = "cfg3_train"
SMI_QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        z = json.load(open(p))
        return dict(hbm_gbs=z["hbm_gbs"], tflops_burst=z["bf16_tflops"], tflops_sustained=z["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops_burst=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region."""

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={SMI_QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path).read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def gemm_flops_forward(cfg):
    """Algorithmic FLOPs of everything the tcgen05 GEMM kernel executes in one forward (projectors, QKV/out/FFN, conv 1-2)."""
    d, ff, N = cfg["hidden_dim"], cfg["dim_feedforward"], cfg["enc_layers"]
    B, Lv, Lt = cfg["batch"], cfg["l_vid"], cfg["l_txt"]
    L = Lv + Lt
    enc = N * (8 * L * d * d + 4 * L * d * ff)
    proj = 2 * Lv * (cfg["v_feat_dim"] * d + d * d) + 2 * Lt * (cfg["t_feat_dim"] * d + d * d)
    conv = 8 * Lv * 3 * d * d
    return B * (enc + proj + conv)


def workload_config(workload, wl, cfg, n_gpus):
    """The `config` object of the JSON line: names the workload only, and is IDENTICAL for --impl b200 and --impl reference (arm
    specific details live in `impl_details`)."""
    return {"workload": workload, "mode": wl["mode"], "batch_per_gpu": cfg["batch"], "global_batch": cfg["batch"] * n_gpus,
            "l_vid": cfg["l_vid"], "l_txt": cfg["l_txt"], "hidden_dim": cfg["hidden_dim"], "nheads": cfg["nheads"],
            "dim_feedforward": cfg["dim_feedforward"], "enc_layers": cfg["enc_layers"], "v_feat_dim": cfg["v_feat_dim"],
            "t_feat_dim": cfg["t_feat_dim"],
            "step": ("forward + criterion + backward + clip_grad_norm(0.1) + AdamW, input_dropout 0.5, droppath 0.1"
                     if wl["mode"] == "train" else "inference forward"),
            "l2_policy": "rotating input batches larger than the 126 MB L2 in total"}


def oracle_step_fn(cfg, mode, batch, device="cpu", dtype=None, autocast=None):
    """One CPU step of the oracle port: forward (mode fwd) or forward + criterion + backward + grad-clip + AdamW (mode train)."""
    from oracle import univtg_oracle as O  # bench.py may execute oracle/ only in the CPU legs

    import contextlib

    sd = {k: v.float().to(device) for k, v in synth.make_state_dict(cfg, seed=0).items()}
    inp = {k: v.to(device) for k, v in synth.make_inputs(cfg, seed=1, batch=batch).items()}
    ctx = (lambda: torch.autocast(device_type="cuda", dtype=autocast)) if autocast is not None else contextlib.nullcontext
    if mode == "fwd":
        def step():
            with torch.no_grad(), ctx():
                return O.forward(sd, cfg, **inp, dtype=torch.float32)["pred_spans"]
        return step
    tgt = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in synth.make_targets(synth.make_inputs(cfg, seed=1, batch=batch), seed=2).items()}
    leaves = {k: v.clone().requires_grad_(not k.startswith("txt_position_embed")) for k, v in sd.items()}
    params = [v for v in leaves.values() if v.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-4)
    wd = {"loss_b": 10.0, "loss_g": 1.0, "loss_f": 10.0, "loss_s_intra": 0.1, "loss_s_inter": 0.1}

    def step():
        with ctx():
            out = O.forward(leaves, cfg, **inp, dtype=torch.float32)
            total = O.weighted_total(O.criterion({k: (v.float() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in out.items()}, tgt), wd)
        opt.zero_grad()
        total.backward()
        torch.nn.utils.clip_grad_norm_(params, 0.1)
        opt.step()
        return total
    return step


def gpu_eager_baseline(cfg, wl, dev, steps=10):
    """The "second bar" of SURVEY.md section 8(d) / BASELINE.md section 3: the reference's fp32 PyTorch path run on the SAME B200
    through torch eager (cuBLAS / ATen kernels) - here the oracle port of that path (oracle/univtg_oracle.py is device-agnostic
    tensor algebra; the reference itself cannot travel to the GPU box).  Three precisions: strict fp32, TF32 matmuls, bf16 autocast.
    A baseline beside the product, never part of it."""
    res = {"what": "oracle port of the reference PyTorch path on this GPU via torch eager", "unit": "pairs/s", "steps": steps}
    B = cfg["batch"]
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    try:
        for name, tf32, ac in (("fp32", False, None), ("tf32", True, None), ("bf16_autocast", True, torch.bfloat16)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            step = oracle_step_fn(cfg, wl["mode"], B, device=dev, autocast=ac)
            for _ in range(3):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            res[name] = {"value": B / (ms * 1e-3), "ms_per_step": ms}
            del step
            torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old_tf32
    return res


def shard_e2e_forward(model, cfg, dev, steps):
    """Inference end to end from a packed fp16 feature shard (univtg_b200/data.py, SURVEY.md section 8 row f-2): the loader assembles
    every padded batch from the memory-mapped shard into pinned buffers and copies it on a side stream one batch ahead; the
    model reads the fp16 features directly; results are read back on the host every step."""
    import tempfile

    import numpy as np

    from univtg_b200 import data as D

    B, Lv, Lt = cfg["batch"], cfg["l_vid"], cfg["l_txt"]
    n_batches = steps + 4
    path = os.path.join(tempfile.gettempdir(), f"univtg_bench_{os.getpid()}.uvshard")
    rng = np.random.default_rng(0)
    vids = [rng.standard_normal((Lv, cfg["v_feat_dim"])).astype(np.float16) * np.float16(0.02) for _ in range(64)]
    qs = [rng.standard_normal((Lt, cfg["t_feat_dim"])).astype(np.float16) * np.float16(0.04) for _ in range(64)]
    samples = [(int(rng.integers(0, 64)), int(rng.integers(0, 64))) for _ in range(B * n_batches)]
    D.write_shard(path, vids, qs, samples)
    try:
        loader = D.ShardLoader(path, batch_size=B, device=dev, slots=3, workers=8)  # direct DMA from the page-locked mapping if allowed
        direct_used, direct_error = bool(loader.direct), getattr(loader, "direct_error", None)
        out_host = [torch.empty(B, Lv).pin_memory() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        model.eval()
        t_ev = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
        seen = 0.0
        with torch.no_grad():
            for i, (batch, _) in enumerate(loader):
                if i == 4:
                    torch.cuda.synchronize()
                    t_ev[0].record()
                out = model(**batch)
                out_host[i % 2].copy_(out["saliency_scores"], non_blocking=True)
                done[i % 2].record()
                if i >= 1:
                    done[(i - 1) % 2].synchronize()
                    seen += float(out_host[(i - 1) % 2][0, 0])
            t_ev[1].record()
            torch.cuda.synchronize()
        ms = t_ev[0].elapsed_time(t_ev[1]) / steps
        loader.close()
        return {"value": B / (ms * 1e-3), "unit": "pairs/s", "ms_per_step": ms, "h2d_bytes_per_step": loader.h2d_bytes(B, Lv, Lt),
                "path": ("copy engines read the page-locked shard mapping directly" if direct_used else "native gather into pinned staging, one H2D per tensor"),
                "direct_refused": direct_error,
                "d2h_bytes_per_step": B * Lv * 4, "what": "forward fed by ShardLoader (packed fp16 shard -> side-stream H2D, one batch ahead)"}
    finally:
        try:
            os.unlink(path)
        except OSError:
            pass


def attention_work(cfg, train):
    """Algorithmic work of the attention core per step: flops 4 L^2 d per sample and layer forward (+ 10 L^2 d backward: five
    contractions), bytes = Q, K, V read + O written as 16-bit (forward; backward reads Q, K, V, dO and writes dQ, dK, dV)."""
    B, L, d, N = cfg["batch"], cfg["l_vid"] + cfg["l_txt"], cfg["hidden_dim"], cfg["enc_layers"]
    fl = 4.0 * L * L * d * B * N
    by = 4.0 * B * L * d * 2 * N
    if train:
        fl += 10.0 * L * L * d * B * N
        by += 7.0 * B * L * d * 2 * N
    return fl, by


def sub_workload(name, dev, operand_format, steps, peaks):
    """A few steps of another BASELINE.json config inside the default run (configs[3] = cfg4_train, configs[4] = cfg5_fwd), with
    the attention kernel's achieved TFLOP/s and HBM GB/s (CUDA events around its launches)."""
    from univtg_b200 import build_model
    from univtg_b200.optim import FlatAdamW

    wl = WORKLOADS[name]
    cfg = synth.CONFIGS[wl["cfg"]]
    train = wl["mode"] == "train"
    model, crit = build_model(synth.reference_args(cfg, device=str(dev), operand_format=operand_format))
    model.load_state_dict(synth.make_state_dict(cfg, seed=0), strict=True)
    model.to(dev)
    crit.to(dev)
    B, Lv, Lt = cfg["batch"], cfg["l_vid"], cfg["l_txt"]
    raw = [synth.make_inputs(cfg, seed=11 + i) for i in range(3)]
    inps = [{k: v.to(dev) for k, v in r.items()} for r in raw]
    if train:
        model.train()
        crit.train()
        opt = FlatAdamW(model, lr=1e-4, weight_decay=1e-4, max_grad_norm=0.1, zero_grad_after_step=True)
        tgts = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in synth.make_targets(r, seed=21 + i).items()} for i, r in enumerate(raw)]

        def step(i):
            out = model(**inps[i % 3])
            total = crit.weighted_total(crit(out, tgts[i % 3]))
            opt.zero_grad()
            total.backward()
            opt.step()
    else:
        model.eval()

        def step(i):
            with torch.no_grad():
                model(**inps[i % 3])
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if train:
        def run():
            out = model(**inps[0])
            crit.weighted_total(crit(out, tgts[0])).backward()
        tl = model.profile_train_step(B, Lv, Lt, run)
    else:
        with torch.no_grad():
            tl = model.profile_forward(inps[0])
    attn_ms = sum(m for k, m in tl if k == 2)
    n_attn = sum(1 for k, m in tl if k == 2)
    gemm_ms = sum(m for k, m in tl if k == 1)
    fl, by = attention_work(cfg, train)
    total_flops, enc_flops = synth.flops_forward(cfg)
    mult = 3 if train else 1
    res = {"workload": name, "ms_per_step": ms, "value": B / (ms * 1e-3), "unit": "pairs/s", "steps": steps,
           "clips_per_s": B * Lv / (ms * 1e-3), "tflops_algorithmic": mult * total_flops / (ms * 1e-3) / 1e12,
           "encoder_tflops_pct_of_sustained_peak": 100.0 * mult * enc_flops / (ms * 1e-3) / 1e12 / peaks["tflops_sustained"],
           "attention": {"launches": n_attn, "ms": attn_ms, "tflops": fl / (attn_ms * 1e-3) / 1e12 if attn_ms > 0 else None,
                         "hbm_gbs_algorithmic": by / (attn_ms * 1e-3) / 1e9 if attn_ms > 0 else None,
                         "frac_of_tensor_peak": fl / (attn_ms * 1e-3) / 1e12 / peaks["tflops_sustained"] if attn_ms > 0 else None,
                         "frac_of_hbm_peak": by / (attn_ms * 1e-3) / 1e9 / peaks["hbm_gbs"] if attn_ms > 0 else None,
                         "flop_per_byte": fl / by},
           "gemm_ms": gemm_ms}
    del model, crit
    torch.cuda.empty_cache()
    return res


def run_reference_arm(args, wl, cfg):
    """CPU arm: the oracle port of the reference's fp32 path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = cfg["batch"]
    cores = pick_threads(oracle_step_fn(cfg, wl["mode"], min(B, 4)))
    step = oracle_step_fn(cfg, wl["mode"], B)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = B * args.steps / dt
    line = {
        "impl": "reference", "metric": "video-query pairs/sec" + (" (fwd+bwd)" if wl["mode"] == "train" else " (fwd)"), "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, wl, cfg, args.gpus),
        "impl_details": {"what": "oracle port of the reference fp32 PyTorch path on the host cores (one process, rank 0)",
                         "batch": B, "threads": cores},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full steps (B={B}) of {args.workload}, oracle/univtg_oracle.py fp32, "
                                   f"torch {torch.__version__} CPU, {cores} threads"},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_json_line(line)


def pick_threads(fn):
    """All host cores the process may use, unless over-subscription (cgroup quota < visible cores) makes fewer threads
    faster: time one call at a few thread counts and keep the best."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (avail, 32, 8) if 1 <= c <= avail}, reverse=True)
    best, best_t = cands[-1], None
    for c in sorted(cands):  # small counts first: a crawling 128-thread run must not eat the time budget
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
        if dt > 20.0:
            break
    torch.set_num_threads(best)
    return best


def cpu_baseline(cfg, wl, workload):
    """Oracle port of the reference fp32 path on the host cores, bounded sample (~10-30 s of CPU work)."""
    sample_b = min(cfg["batch"], 8)
    step = oracle_step_fn(cfg, wl["mode"], sample_b)
    cores = pick_threads(step)
    t0 = time.perf_counter()
    n = 0
    while True:
        step()
        n += 1
        dt = time.perf_counter() - t0
        if dt > 10.0 or n >= 50:
            break
    return {"value": sample_b * n / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": f"{n} steps of B={sample_b} ({workload} shape, mode {wl['mode']}), oracle/univtg_oracle.py fp32 on {cores} "
                      f"torch threads"}


def gemm_traffic_bytes():
    """DRAM bytes (read + write) per launch of the GEMM kernel from the committed `ncu --set full` capture (mean over the 58
    launches of one train step; profiles/gemm_traffic.json), or None when the file is absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "gemm_traffic.json")) as f:
            return int(json.load(f)["bytes_per_launch_mean"])
    except Exception:
        return None


def grad_sync_check(dist, dev, rank, world, operand_format, overlap):
    """Hardware check of the data-parallel exchange (SURVEY.md 8e: every loss is a LOCAL-batch mean, so the reference semantics is
    DDP's average of the ranks' gradients): on a small config every rank back-propagates its own batch through the overlapped
    exchange; rank r then recomputes all `world` batches alone (no exchange) and averages.  Reports the relative L2 difference."""
    from univtg_b200 import build_model, ddp

    cfg = dict(synth.CONFIGS["tiny"], nheads=2)
    results = []
    for mode in ("exchange", "local"):
        model, crit = build_model(synth.reference_args(cfg, device=str(dev), operand_format=operand_format, droppath=0.0, input_dropout=0.0))
        model.load_state_dict(synth.make_state_dict(cfg, seed=5), strict=True)
        model.to(dev).train()
        crit.to(dev).train()
        model.direct_grad = True
        if mode == "exchange":
            ddp.attach_flat_allreduce(model, overlap=overlap)
        acc = None
        for r in ([rank] if mode == "exchange" else range(world)):
            raw = synth.make_inputs(cfg, seed=900 + r, ragged=True, batch=4)
            tgt = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in synth.make_targets(raw, seed=950 + r).items()}
            model.__dict__["_flat_grad_dirty"] = False
            out = model(**{k: v.to(dev) for k, v in raw.items()})
            crit.weighted_total(crit(out, tgt)).backward()
            torch.cuda.synchronize()
            flat = model._grad_buffer()[0].clone()
            acc = flat if acc is None else acc + flat
        results.append(acc / (1 if mode == "exchange" else world))
        ddp.detach_flat_allreduce(model)
        del model, crit
    rel = float((results[0] - results[1]).norm() / results[1].norm().clamp_min(1e-30))
    t = torch.tensor([rel], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # fp32 atomics in split-K reductions + NCCL's reduction order: a few 1e-4 relative at most
    return {"what": "all-reduced gradient vs the average of the ranks' gradients recomputed on one GPU (tiny config, B=4 per rank)",
            "grad_rel_err": float(t[0]), "tolerance": 2e-3, "world": world}


def ddp_cfg4_point(dist, dev, rank, world, operand_format, overlap, steps=10):
    """BASELINE.json configs[3]: the vlp_ddp pre-training shape (B = 32 per rank, L_v = 150) through the same exchange; a few steps."""
    from univtg_b200 import build_model, ddp
    from univtg_b200.optim import FlatAdamW

    cfg = synth.CONFIGS["cfg4"]
    model, crit = build_model(synth.reference_args(cfg, device=str(dev), operand_format=operand_format))
    model.load_state_dict(synth.make_state_dict(cfg, seed=0), strict=True)
    model.to(dev).train()
    crit.to(dev).train()
    opt = FlatAdamW(model, lr=1e-4, weight_decay=1e-4, max_grad_norm=0.1, zero_grad_after_step=True)
    ddp.broadcast_parameters(model)
    ddp.attach_flat_allreduce(model, overlap=overlap)
    raws = [synth.make_inputs(cfg, seed=31 + 7 * rank + i) for i in range(3)]
    inps = [{k: v.to(dev) for k, v in r.items()} for r in raws]
    tgts = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in synth.make_targets(r, seed=61 + i).items()} for i, r in enumerate(raws)]

    def step(i):
        out = model(**inps[i % 3])
        total = crit.weighted_total(crit(out, tgts[i % 3]))
        opt.zero_grad()
        total.backward()
        opt.step()
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0]) / steps
    B = cfg["batch"]
    del model, crit, opt
    torch.cuda.empty_cache()
    return {"workload": "cfg4_train", "global_batch": B * world, "l_vid": cfg["l_vid"], "ms_per_step": ms,
            "value": B * world / (ms * 1e-3), "unit": "pairs/s", "steps": steps, "timing": "CUDA events, max over ranks"}


_REAL_STDOUT_FD = None


def _quiet_stdout():
    """stdout must carry exactly ONE JSON line: until it is printed, file descriptor 1 points at stderr so that banners written
    by native libraries (e.g. "NCCL version ..." at communicator creation) cannot precede it."""
    global _REAL_STDOUT_FD
    if _REAL_STDOUT_FD is None:
        sys.stdout.flush()
        _REAL_STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json_line(line):
    sys.stdout.flush()
    if _REAL_STDOUT_FD is not None:
        os.dup2(_REAL_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)


DUMP_PARAM_SAMPLE = 1 << 20  # parameters written by --dump-outputs: a fixed, seeded sample of this many elements


def dump_outputs(path, model, last, train):
    """Writes what the last timed step returned, as .npy files (about 22 MB for the default workload): the model outputs of its
    batch, and for a train step also its five losses, the weighted total and a fixed sample of the updated parameters (state_dict
    order).  Inputs and random draws are seeded, so two builds run with the same arguments can be compared file by file.  The
    backward's split-K reductions add in fp32 atomics, so train-mode files of two runs agree to a tolerance, not bit for bit
    (measured on one B200 at 1000 W, 20 steps after 5 warm-up: parameters within 1.1e-3, outputs within 6.1e-3 absolute)."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    out = last["out"]
    arrays = {k: out[k] for k in ("pred_logits", "pred_spans", "saliency_scores", "vid_mem_proj", "txt_mem_proj")}
    if train:
        arrays.update({k: v for k, v in last["losses"].items()})
        arrays["loss_total"] = last["total"]
        flat = torch.nn.utils.parameters_to_vector(model.parameters())
        g = torch.Generator().manual_seed(0)
        idx = torch.randint(0, flat.numel(), (min(DUMP_PARAM_SAMPLE, flat.numel()),), generator=g).sort().values
        arrays["params_sample"] = flat[idx.to(flat.device)]
        arrays["params_sample_index"] = idx.double()
    for k, v in arrays.items():
        v = v.detach().cpu()
        np.save(os.path.join(path, k + ".npy"), (v if v.dtype == torch.float64 else v.float()).numpy())


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--operand-format", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graphs", action="store_true",
                    help="inference workloads: replay the forward from a CUDA graph (default: eager launches chained by "
                         "programmatic dependent launch, which measured faster: 0.712 vs 0.735 ms at cfg2)")
    ap.add_argument("--no-overlap", action="store_true", help="N>1: one all-reduce after the backward instead of stage slices")
    ap.add_argument("--train-graph-probe", action="store_true",
                    help="experiment: also time the train step replayed from ONE CUDA graph (host launch cost removed; RNG seed and "
                         "AdamW step count frozen at capture time, so this is a timing probe, not a training mode)")
    ap.add_argument("--static-loss-scale", action="store_true", help="fixed fp16 loss scale (no overflow flag read-back)")
    ap.add_argument("--no-zero-after-step", action="store_true",
                    help="zero the flat gradient buffer in front of the backward instead of on a side stream behind the optimizer step")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra legs of the default line (cfg4_train / cfg5_fwd sub-results, GPU torch-eager baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, sample indices float64; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    torch.manual_seed(0)  # the dropout / DropPath seeds are drawn from torch's CPU generator
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload]
    cfg = synth.CONFIGS[wl["cfg"]]
    train = wl["mode"] == "train"

    if args.impl == "reference":
        run_reference_arm(args, wl, cfg)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a GPU (no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        # stdout carries exactly one JSON line: NCCL's own banner ("NCCL version ...", printed when NCCL_DEBUG is set) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        # the gradient all-reduce overlaps the backward: cap the SMs its kernels take (the backward's persistent GEMM grids are
        # sized for what is left, univtg_b200/ddp.py: UNIVTG_DDP_SM_RESERVE)
        os.environ.setdefault("NCCL_MAX_CTAS", "32")
        os.environ.setdefault("UNIVTG_DDP_SM_RESERVE", os.environ["NCCL_MAX_CTAS"])
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    from univtg_b200 import build_model, ddp

    model, crit = build_model(synth.reference_args(cfg, device=str(dev), operand_format=args.operand_format))
    model.load_state_dict(synth.make_state_dict(cfg, seed=0), strict=True)
    model.to(dev)
    crit.to(dev)
    B, Lv, Lt, d = cfg["batch"], cfg["l_vid"], cfg["l_txt"], cfg["hidden_dim"]
    opt = None
    if train:
        model.train()
        crit.train()
        # the reference's update (main/config.py:349-350 AdamW; train_vlp_ddp.py:66-68 clip 0.1 + step) fused over the flat
        # parameter / gradient buffers: univtg_adamw_step, two launches per step
        from univtg_b200.optim import FlatAdamW
        opt = FlatAdamW(model, lr=1e-4, weight_decay=1e-4, max_grad_norm=0.1, dynamic_loss_scale=not args.static_loss_scale,
                        zero_grad_after_step=not args.no_zero_after_step)
        if dist is not None:
            ddp.broadcast_parameters(model)
            # NCCL all-reduce of the flat gradient buffer, issued in backward-stage slices on a side stream (overlaps backward)
            ddp.attach_flat_allreduce(model, overlap=not args.no_overlap)
    else:
        model.eval()
        model.use_cuda_graphs = bool(args.graphs)  # the 41 launches of a forward replayed from one CUDA graph per shape

    # Rotating set of distinct input batches whose total size exceeds the 126 MB L2 (no L2-resident inputs between steps).
    per_batch = B * (Lv * cfg["v_feat_dim"] + Lt * cfg["t_feat_dim"] + Lv + Lt) * 4
    n_rot = max(2, int(160e6 // per_batch) + 1)
    host_batches, host_targets = [], []
    for i in range(n_rot):
        inp = synth.make_inputs(cfg, seed=1 + 7 * rank + i)
        host_batches.append({k: v.pin_memory() for k, v in inp.items()})
        if train:
            host_targets.append({k: v.pin_memory() for k, v in synth.make_targets(inp, seed=100 + 7 * rank + i).items()})
    dev_batches = [{k: v.to(dev) for k, v in hb.items()} for hb in host_batches]
    dev_targets = [{k: v.to(dev) for k, v in ht.items()} for ht in host_targets]
    from univtg_b200 import _lib as uvlib
    lib = uvlib.load_library()

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def train_step(inputs, targets, keep=None):
        out = model(**inputs)
        ld = crit(out, targets)
        total = crit.weighted_total(ld)  # = sum(ld[k] * weight_dict[k]) of the reference loop, as one dot product
        opt.zero_grad(set_to_none=True)
        total.backward()
        opt.step()  # clip_grad_norm_(0.1) (reference --grad_clip 0.1) + AdamW
        if keep is not None:
            keep.update(out=out, losses=ld, total=total)
        return total

    def device_step(i, keep=None):
        if train:
            return train_step(dev_batches[i % n_rot], dev_targets[i % n_rot], keep)
        with torch.no_grad():
            out = model(**dev_batches[i % n_rot])
        if keep is not None:
            keep["out"] = out
        return out

    # ------------------------------------------------ device-resident timing ------------------------------------------------
    for i in range(args.warmup):
        device_step(i)
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    last = {} if args.dump_outputs else None  # what each timed step returned; the last one is written out below
    launches0 = int(lib.univtg_launch_count())
    e0.record()
    for i in range(args.steps):
        device_step(i, last)
    e1.record()
    sync_all()
    ms_total = e0.elapsed_time(e1)
    gpu_launches = int(lib.univtg_launch_count()) - launches0  # kernels of THIS library launched inside the timed region
    if last is not None and rank == 0:
        dump_outputs(args.dump_outputs, model, last, train)
    last = None
    # host side of the same loop: how long the CPU needs to ENQUEUE a step (5 steps = ~600 launches stay below the driver's launch
    # queue depth, so the host is not throttled by the GPU here).  enqueue time ~ ms_per_step means the step is host-bound.
    sync_all()
    t_h0 = time.perf_counter()
    for i in range(5):
        device_step(i)
    host_enqueue_ms = (time.perf_counter() - t_h0) * 1e3 / 5
    sync_all()

    # -------------------------------------------- end-to-end through the public API ------------------------------------
    # Every step copies ITS inputs from pinned host memory and reads ITS result back on the host.  The H2D copy of step
    # i+1 is issued on a side stream while step i computes (two staging slots) - the pipelining any input loop would do.
    n_slot = 2
    stage = [{k: torch.empty_like(v, device=dev) for k, v in host_batches[0].items()} for _ in range(n_slot)]
    stage_t = [{k: torch.empty_like(v, device=dev) for k, v in host_targets[0].items()} if train else {} for _ in range(n_slot)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(n_slot)]   # staging slot filled
    freed = [torch.cuda.Event() for _ in range(n_slot)]   # staging slot consumed by compute
    if train:
        out_host = [{"loss": torch.empty(()).pin_memory()} for _ in range(2)]
    else:
        out_host = [{"pred_logits": torch.empty(B, Lv, 1).pin_memory(), "pred_spans": torch.empty(B, Lv, 2).pin_memory(),
                     "saliency_scores": torch.empty(B, Lv).pin_memory()} for _ in range(2)]

    def issue_copy(i):
        slot = i % n_slot
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[slot])
            hb = host_batches[i % n_rot]
            for k in stage[slot]:
                stage[slot][k].copy_(hb[k], non_blocking=True)
            if train:
                ht = host_targets[i % n_rot]
                for k in stage_t[slot]:
                    stage_t[slot][k].copy_(ht[k], non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_run(n):
        """Host loop with one step of look-ahead: step i+1 is enqueued before the host blocks on step i's result, so the GPU
        never waits for Python.  Every step still copies ITS inputs from pinned host memory and ITS result is read on the host
        (result buffers are double-buffered; `seen` receives each step's value)."""
        main = torch.cuda.current_stream()
        for s_ in range(n_slot):
            freed[s_].record(main)
        issue_copy(0)
        done = [torch.cuda.Event() for _ in range(2)]
        seen = []
        for i in range(n):
            slot = i % n_slot
            if i + 1 < n:
                issue_copy(i + 1)
            main.wait_event(ready[slot])
            hb = out_host[i % 2]
            if train:
                total = train_step(stage[slot], stage_t[slot])
                hb["loss"].copy_(total.detach(), non_blocking=True)  # the reference logs float(losses) every step
            else:
                with torch.no_grad():
                    out = model(**stage[slot])
                for k, hbuf in hb.items():
                    hbuf.copy_(out[k], non_blocking=True)
            freed[slot].record(main)
            done[i % 2].record(main)
            if i >= 1:  # consume step i-1's result on the host while step i runs
                done[(i - 1) % 2].synchronize()
                prev = out_host[(i - 1) % 2]
                seen.append(float(prev["loss"]) if train else float(prev["saliency_scores"][0, 0]))
        if n >= 1:
            done[(n - 1) % 2].synchronize()
            last = out_host[(n - 1) % 2]
            seen.append(float(last["loss"]) if train else float(last["saliency_scores"][0, 0]))
        return seen

    e2e_run(3)
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    e2e_run(args.steps)
    f1.record()
    sync_all()
    ms_e2e = f0.elapsed_time(f1)
    clocks = sampler.stop() if rank == 0 else None

    # ------------------- forward-only (inference) throughput on the same shapes, reported beside a train workload -----------
    fwd_only = None
    if train:
        model.eval()
        model.use_cuda_graphs = bool(args.graphs)
        with torch.no_grad():
            for i in range(3):
                model(**dev_batches[i % n_rot])
            sync_all()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for i in range(args.steps):
                model(**dev_batches[i % n_rot])
            g1.record()
            sync_all()
        ms_fwd = g0.elapsed_time(g1)
        fwd_only = {"value": B * args.steps * n_gpus / (ms_fwd * 1e-3), "unit": "pairs/s", "ms_per_step": ms_fwd / args.steps,
                    "note": "BASELINE configs[1]: inference forward on the same shapes (max over ranks not applied)"}
        if n_gpus == 1 and not args.no_extras:
            try:
                fwd_only["e2e_from_feature_shard"] = shard_e2e_forward(model, cfg, dev, args.steps)
            except Exception as ex:
                fwd_only["e2e_from_feature_shard"] = {"error": repr(ex)[:300]}
        model.use_cuda_graphs = False
        model.train()

    # ------------------- decode + temporal NMS of the evaluation loop (SURVEY section 8 rows a16 / f-1), inference workloads ----------
    postproc_line = None
    if not train and rank == 0:
        from univtg_b200 import postproc as pp
        durs = [150.0] * B
        ts = ((torch.arange(Lv, dtype=torch.float32, device=dev) + 0.5) / Lv)[None, :, None].expand(B, Lv, 2).contiguous()
        with torch.no_grad():
            out = model(**dev_batches[0])
        tgt = {"timestamp": ts, "timestamp_mask": dev_batches[0]["src_vid_mask"]}

        def post():
            dec = pp.decode_mr(out, tgt, durs)
            return dec, pp.temporal_nms(dec["windows_r4"], 0.7, 10, 10)
        for _ in range(3):
            post()
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(20):
            dec, _ = post()
        p1.record()
        torch.cuda.synchronize()
        gpu_us = p0.elapsed_time(p1) / 20 * 1e3
        from oracle import postproc_oracle as PO  # CPU leg: the reference's Python decode + NMS on the same outputs
        cpu_out = {k: out[k].cpu() for k in ("pred_logits", "pred_spans")}
        t0 = time.perf_counter()
        rows = PO.decode_mr(cpu_out["pred_logits"], cpu_out["pred_spans"], ts.cpu(), tgt["timestamp_mask"].cpu(), durs)
        PO.post_processing_mr_nms(rows, 0.7, 10, 10)
        cpu_ms = (time.perf_counter() - t0) * 1e3
        postproc_line = {"what": "decode_mr + temporal_nms(0.7, 10, 10) on one batch", "gpu_us_per_batch": gpu_us,
                         "cpu_port_ms_per_batch": cpu_ms, "bit_exact_vs_port": bool(dec["windows_r4"].cpu().tolist() == rows)}

    # ------------------- per-kernel-class durations (CUDA events around the launches of the measured step) ---------------------
    # train workloads: the WHOLE step's GEMM launches (forward + dgrad + wgrad), inference workloads: the forward's
    kind_ms = {0: [], 1: [], 2: [], 3: []}
    n_kind = {0: 0, 1: 0, 2: 0, 3: 0}
    if train:
        for i in range(5):
            def run(i=i):
                out = model(**dev_batches[i % n_rot])
                total = crit.weighted_total(crit(out, dev_targets[i % n_rot]))
                opt.zero_grad(set_to_none=True)
                total.backward()
            tl = model.profile_train_step(B, Lv, Lt, run)
            acc = {0: 0.0, 1: 0.0, 2: 0.0, 3: 0.0}
            n_kind = {0: 0, 1: 0, 2: 0, 3: 0}
            for kind, ms in tl:
                acc[kind] += ms
                n_kind[kind] += 1
            for k in acc:
                kind_ms[k].append(acc[k])
    else:
        was_training = model.training
        model.eval()
        with torch.no_grad():
            for i in range(5):
                tl = model.profile_forward(dev_batches[i % n_rot])
                acc = {0: 0.0, 1: 0.0, 2: 0.0, 3: 0.0}
                n_kind = {0: 0, 1: 0, 2: 0, 3: 0}
                for kind, ms in tl:
                    acc[kind] += ms
                    n_kind[kind] += 1
                for k in acc:
                    kind_ms[k].append(acc[k])
        model.train(was_training)
    gemm_ms = statistics.median(kind_ms[1])
    attn_ms = statistics.median(kind_ms[2])
    row_ms = statistics.median(kind_ms[0]) + statistics.median(kind_ms[3])

    # ------------------- extra legs of the default line (rank 0 of a single-GPU run) --------------------------------------------
    extras = {}
    if n_gpus == 1 and not args.no_extras and args.workload == DEFAULT_WORKLOAD:
        peaks_x = load_peaks()
        dev_batches.clear()
        dev_targets.clear()
        torch.cuda.empty_cache()
        try:
            extras["cfg4_train"] = sub_workload("cfg4_train", dev, args.operand_format, 10, peaks_x)
            extras["cfg5_fwd"] = sub_workload("cfg5_fwd", dev, args.operand_format, 10, peaks_x)
        except Exception as ex:  # never lose the headline to an extra leg
            extras["error"] = repr(ex)[:300]
        try:
            extras["gpu_eager_baseline"] = gpu_eager_baseline(cfg, wl, dev)
        except Exception as ex:
            extras["gpu_eager_baseline"] = {"error": repr(ex)[:300]}

    graph_probe = None
    if train and args.train_graph_probe and dist is None:
        try:
            opt.dynamic_loss_scale = False  # its flag read-back synchronises with the host
            opt.zero_grad_after_step = False  # a side-stream fill joined by the NEXT step cannot live inside a one-step capture
            model.__dict__.pop("_flat_grad_prezeroed", None)
            inp0 = {k: v.to(dev) for k, v in host_batches[0].items()}
            tgt0 = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in host_targets[0].items()}
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    train_step(inp0, tgt0)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                train_step(inp0, tgt0)
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            for _ in range(args.steps):
                graph.replay()
            q1.record()
            torch.cuda.synchronize()
            ms_g = q0.elapsed_time(q1) / args.steps
            graph_probe = {"ms_per_step": ms_g, "value": B / (ms_g * 1e-3), "note": "one CUDA graph per step, same batch every replay"}
        except Exception as ex:
            graph_probe = {"error": repr(ex)[:400]}

    # ------------------- N > 1: is the exchanged gradient the average of the ranks' gradients, and did the replicas stay equal? ----
    sync_check = None
    cfg4_line = None
    if dist is not None and train:
        sync_check = grad_sync_check(dist, dev, rank, world, args.operand_format, not args.no_overlap)
        flat_p = opt._flat_p
        cs = torch.stack([flat_p.double().sum(), flat_p.double().abs().sum()])
        gathered = [torch.zeros_like(cs) for _ in range(world)]
        dist.all_gather(gathered, cs)
        same = all(bool(torch.equal(gathered[0], g_)) for g_ in gathered)
        sync_check["param_checksum_equal_across_ranks"] = same
        sync_check["status"] = "ok" if (same and sync_check["grad_rel_err"] <= sync_check["tolerance"]) else "MISMATCH"
        if args.workload == DEFAULT_WORKLOAD and not args.no_extras:
            cfg4_line = ddp_cfg4_point(dist, dev, rank, world, args.operand_format, not args.no_overlap)

    # max over ranks
    t = torch.tensor([ms_total, ms_e2e], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(t[0]), float(t[1])

    if rank == 0:
        peaks = load_peaks()
        pairs = B * args.steps * n_gpus
        value = pairs / (ms_total * 1e-3)
        e2e_value = pairs / (ms_e2e * 1e-3)
        total_flops, enc_flops = synth.flops_forward(cfg)
        if train:
            total_flops, enc_flops = 3 * total_flops, 3 * enc_flops  # dgrad + wgrad
        gflops = gemm_flops_forward(cfg) * (3 if train else 1)  # train: forward + dgrad + wgrad launches of the same kernel
        n_gemm = max(1, n_kind[1])
        achieved_tf = gflops / (gemm_ms * 1e-3) / 1e12
        h2d = sum(v.numel() * v.element_size() for v in host_batches[0].values())
        if train:
            h2d += sum(v.numel() * v.element_size() for v in host_targets[0].values())
        d2h = sum(v.numel() * v.element_size() for v in out_host[0].values())
        step_ms = ms_total / args.steps
        line = {
            "metric": "video-query pairs/sec" + (" (fwd+bwd)" if train else " (fwd)"), "value": value, "unit": "pairs/s",
            "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16" if args.operand_format == "fp16" else "bf16",
            "data": "synthetic",
            "config": workload_config(args.workload, wl, cfg, n_gpus),
            "impl_details": {
                "operands": "fp16 activations/weights/gradients (gradients under a 2^10 loss scale), f32 accumulate + statistics + master weights",
                "step": ("forward + criterion + backward + clip_grad_norm(0.1) + AdamW; dropout / DropPath multipliers generated in-kernel (Philox); the flat gradient buffer is zero-filled on a side stream behind the update (FlatAdamW zero_grad_after_step)" if train
                         else ("forward (launches chained by programmatic dependent launch)" if (not args.graphs)
                               else "forward (CUDA-graph replay)")),
                "parallelism": (f"dp{n_gpus}: shard by sample; flat fp32 gradient buffer NCCL all-reduced (AVG) in backward-stage slices on a side stream" if train
                                else f"replicas x{n_gpus} (shard by sample, no collective)"),
                "l2_policy": f"{n_rot} rotating input batches ({n_rot * per_batch / 1e6:.0f} MB > 126 MB L2)",
                "clips_per_s": value * Lv},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "host_enqueue_ms_per_step": host_enqueue_ms,
            "gpu_launches": gpu_launches,
            "launches_per_step": gpu_launches / args.steps,
            "clocks": clocks,
            "tflops_algorithmic": total_flops / (step_ms * 1e-3) / 1e12,
            "encoder_tflops_pct_of_sustained_peak": 100.0 * enc_flops / (step_ms * 1e-3) / 1e12 / peaks["tflops_sustained"],
            "roofline": {"kernel": "gemm_tcgen05_kernel", "bound": "tensor", "achieved": achieved_tf,
                         "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": achieved_tf / peaks["tflops_sustained"],
                         "traffic": gemm_traffic_bytes(),
                         "traffic_source": "static: mean DRAM read+write bytes per launch over the 58 GEMM launches of one train step in the committed ncu --set full capture (profiles/gemm_traffic.json), not measured in this run",
                         "peak_source": peaks["source"] + ", sustained (kernel timed inside a step)",
                         "scope": ("every launch of the kernel in the train step: forward + dgrad + wgrad (CUDA events around each launch)" if train
                                   else "forward launches of the kernel (CUDA events between launches)"),
                         "launches_per_step": n_gemm, "avg_launch_us": gemm_ms / n_gemm * 1e3,
                         "flops_per_launch": gflops / n_gemm,
                         "step_share": {"gemm_ms": gemm_ms, "attention_ms": attn_ms, "row_kernels_ms": row_ms}},
        }
        if fwd_only is not None:
            line["forward_only"] = fwd_only
        if postproc_line is not None:
            line["postproc"] = postproc_line
        for k_, v_ in extras.items():
            line[k_] = v_
        if graph_probe is not None:
            line["train_graph_probe"] = graph_probe
        if sync_check is not None:
            line["grad_sync_check"] = sync_check["status"]
            line["grad_sync_detail"] = sync_check
        if cfg4_line is not None:
            line["cfg4_train"] = cfg4_line
        if n_gpus == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(cfg, wl, args.workload)
        emit_json_line(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
