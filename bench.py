#!/usr/bin/env python
"""Benchmark of the CLIP-ViP video-text hot path (BASELINE.json metric: video-text pairs/s, 12f x 224^2, 32 tok).

One "step" = one pass of the hot path over one batch of synthetic input:
    VidCLIP forward (video tower + text tower)  ->  embedding all-gather + in-batch InfoNCE (learnable temperature)
    ->  backward through both towers (all parameter gradients)  ->  (N > 1) data-parallel gradient averaging.
Workload = BASELINE.json configs[1] per GPU: ViT-B/16, 12 frames x 224^2, 32 tokens, batch 64 per GPU, bf16 compute
with fp32 master parameters / fp32 gradients, random-init weights of the reference's init statistics, synthetic data.

    python bench.py --gpus N --steps K --warmup W            # this repo (N > 1: launched under torchrun, NCCL)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs as DIR/*.npy

Prints ONE JSON line (rank 0).  `value` = pairs/s with inputs resident in HBM (CUDA-event timed, max over ranks);
`e2e` = the same through the public module API with pinned HOST buffers (prefetched H2D of every step's inputs and
a D2H read of the loss inside the timed region); `roofline` = the tcgen05 GEMM kernel's achieved TFLOP/s over all of
its launches in one step (CUDA events around each launch) against MEASURED_PEAKS.json; `cpu_baseline` = the oracle
timed on this box's host cores on a bounded sample.
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

METRIC = "video-text pairs/sec (12f x 224^2, 32 tok), CLIP-ViP ViT-B/16 fwd+InfoNCE+bwd"
UNIT = "pairs/s"
T_FRAMES, L_TOK, PER_GPU_BATCH = 12, 32, 64


def flop_model():
    from oracle import clipvip_oracle as O     # FLOP accounting only (BASELINE.md §2), never on the product path
    return O.flops_per_pair(O.ClipVipCfg(), T_FRAMES, L_TOK)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"tflops": float(p.get("bf16_tflops_sustained", p.get("bf16_tflops"))), "hbm_gbs": float(p["hbm_gbs"]),
                "source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)"}
    return {"tflops": 1400.0, "hbm_gbs": 6650.0, "source": "B200_PROFILING.md fallback, sustained (of fallback)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        sm, smax, power, reasons = [], None, [], set()
        for line in self.tmp.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); smax = float(parts[2]); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.tmp.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_SAMPLE = 1 << 22     # float32 elements kept of a larger output (16 MB); at most four outputs are dumped per run


def flat_grads(params):
    """Every parameter gradient of the last step, flattened and concatenated in parameter order (zeros where none was made)."""
    import torch
    return torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1).float() for p in params])


def dump_outputs(path, arrays):
    """--dump-outputs: write each array as <path>/<name>.npy in float32.  An array of more than DUMP_SAMPLE elements is replaced
    by its flattened elements at DUMP_SAMPLE indices drawn from a fixed seed (sorted, duplicates dropped), the same in every run,
    so that two builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).unique()
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace
    from xpretrain_b200 import ops
    from xpretrain_b200.modeling import VidCLIP
    from xpretrain_b200.optimization.loss import gather_nce_loss
    from xpretrain_b200.utils import distributed as xdist

    # N > 1, optional (XP_SM_RESERVE=n, default 0): cap NCCL at n CTAs and leave n SMs out of every backward GEMM grid so that the
    # overlapped gradient all-reduce never displaces a persistent GEMM CTA.  Measured: +2.8 % at 2 GPUs, but -2.6 % at 8 GPUs, where
    # the thinner all-reduce (1.75x the bytes per rank) exposes its tail (profiles/r02_bench_n8_*.json) — hence off by default.
    reserve = int(os.environ.get("XP_SM_RESERVE", "0")) if int(os.environ.get("WORLD_SIZE", "1")) > 1 else 0
    if reserve > 0:
        os.environ.setdefault("NCCL_MAX_CTAS", str(reserve))
    rank, local, world = xdist.init_from_env("nccl")
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
    # (the reservation is applied by the model during backward only: model.clipmodel.nccl_sm_reserve below)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B, T, Lt = args.batch, T_FRAMES, L_TOK

    add = SimpleNamespace(type="ViP", temporal_size=12, if_use_temporal_embed=1, logit_scale_init_value=4.60, add_cls_num=3)
    torch.manual_seed(0)
    model = VidCLIP(SimpleNamespace(clip_config="openai/clip-vit-base-patch16", clip_weights="",
                                    clip_vision_additional_config=add))
    with torch.no_grad():
        model.clipmodel.vision_model.embeddings.temporal_embedding.normal_(0, 0.02)
    model = model.to(dev)
    params = [p for p in model.parameters()]
    if world > 1:   # DP gradient averaging overlapped with backward (logit_scale's gradient is identical on all ranks)
        comm = torch.bfloat16 if os.environ.get("XP_GRAD_COMM", "fp32") == "bf16" else None
        model.clipmodel.grad_ready_hook = xdist.OverlappedGradAverager(comm_dtype=comm)
        model.clipmodel.nccl_sm_reserve = reserve

    # synthetic inputs (SURVEY.md §8d): pinned host copies for the e2e leg, device copies for the resident leg
    g = torch.Generator().manual_seed(1234 + rank)
    n_host = 2
    host = []
    for _ in range(n_host):
        v = torch.randn(B, T, 3, 224, 224, generator=g).pin_memory()
        ids = torch.randint(1, 49406, (B, Lt), generator=g)
        ids[:, -1] = 49407
        host.append((v, ids.pin_memory(), torch.ones(B, Lt, dtype=torch.long).pin_memory()))
    resident = [tuple(t.to(dev) for t in h) for h in host]

    last_step = {}

    def step(video, ids, mask):
        for p in params:
            p.grad = None
        out = model(video=video, text_input_ids=ids, text_input_mask=mask)
        loss = gather_nce_loss(out["vis_features"], out["text_features"], model.clipmodel.logit_scale)
        loss.backward()
        last_step.update(loss=loss.detach(), vis=out["vis_features"].detach(), txt=out["text_features"].detach())
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps between barrier+synchronize on both sides; CUDA-event time, max over ranks (ms per step)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    for i in range(args.warmup):
        step(*resident[i % n_host])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms_resident = timed(lambda i: step(*resident[i % n_host]), args.steps)
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:         # before the legs below overwrite the gradients
        dump_outputs(args.dump_outputs, {"loss": last_step["loss"], "vis_features": last_step["vis"],
                                         "text_features": last_step["txt"], "param_grads": flat_grads(params)})

    # ---- e2e: host buffers -> prefetched H2D on a side stream (the reference's PrefetchLoader pattern,
    #      dataloader.py:92-157) -> module API -> loss.item() (D2H) every step
    copy_stream = torch.cuda.Stream()
    slots = [None, None]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            slots[i % 2] = tuple(t.to(dev, non_blocking=True) for t in host[i % n_host])
            ev = torch.cuda.Event(); ev.record(copy_stream)
        return ev

    last = {"loss": None}

    def e2e_loop(steps):
        ev = prefetch(0)
        for i in range(steps):
            torch.cuda.current_stream().wait_event(ev)
            batch = slots[i % 2]
            for t in batch:
                t.record_stream(torch.cuda.current_stream())
            if i + 1 < steps:
                ev = prefetch(i + 1)
            last["loss"] = step(*batch).detach().item()   # device -> host read of the step's result

    e2e_loop(2)                                            # warm the copy path
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_loop(args.steps)
    e1.record()
    barrier()
    ms_t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_t) / args.steps
    h2d = sum(t.numel() * t.element_size() for t in host[0])

    # ---- extra (SURVEY.md §8f.4): the same e2e loop fed with the decoder's uint8 [B, T, H, W, 3] frames — the reference's
    #      `/255` + Normalize runs inside the patch-extraction kernel, a step uploads 1 byte per sample value instead of 4
    e2e_u8 = None
    if world == 1:
        gu = torch.Generator().manual_seed(99)
        host_u8 = [(torch.randint(0, 256, (B, T, 224, 224, 3), dtype=torch.uint8, generator=gu).pin_memory(), h[1], h[2])
                   for h in host]
        host_f32, host[:] = list(host), host_u8
        e2e_loop(2)
        barrier()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        e2e_loop(args.steps)
        u1.record()
        barrier()
        ms_u8 = u0.elapsed_time(u1) / args.steps
        e2e_u8 = {"what": "module API, pinned uint8 HWC frames (preprocessing fused into the patch extraction) + loss.item() per step",
                  "value": round(B / ms_u8 * 1e3, 2), "unit": UNIT, "ms_per_step": round(ms_u8, 3),
                  "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host_u8[0]), "d2h_bytes_per_step": 4}
        host[:] = host_f32
        del host_u8

    # ---- roofline of the dominant kernel (the tcgen05 GEMM): CUDA events around every launch of one step
    roof = None
    # per-launch / per-block CUDA-event timings below are taken with the text tower and the bias column sums on the MAIN stream:
    # kernels that overlap on side streams would be charged each other's time
    model.clipmodel.overlap_text_tower = model.clipmodel.overlap_colsum = False
    if rank == 0 or world > 1:
        rec = []
        ops.set_gemm_timer(rec)
        step(*resident[0])
        torch.cuda.synchronize()
        ops.set_gemm_timer(None)
        g_ms = sum(e0_.elapsed_time(e1_) for (_, e0_, e1_) in rec)
        g_flops = sum(f for (f, _, _) in rec)
        peaks = measured_peaks()
        achieved = g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
        roof = {"kernel": "xp::gemm_kernel (tcgen05 bf16, all launches of one step)", "bound": "tensor",
                "achieved": round(achieved, 1), "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": round(achieved / peaks["tflops"], 4), "traffic": ncu_traffic()[0],
                "traffic_of": ncu_traffic()[1], "peak_source": peaks["source"],
                "launches_per_step": len(rec), "gemm_ms_per_step": round(g_ms, 3),
                "gemm_share_of_step": round(g_ms / ms_resident, 4)}

    # ---- BASELINE.json metric (2): ViT-block %-of-tensor-roofline — CUDA events around each of the 12 ViP blocks
    #      (QKV + proxy-token attention + out-proj + MLP, K3-K8) of one un-instrumented step, fwd and fwd+bwd
    vit_block = None
    if rank == 0 or world > 1:
        blk = []
        model.clipmodel.block_timer = blk
        step(*resident[0])
        torch.cuda.synchronize()
        model.clipmodel.block_timer = None
        f_ms = [a.elapsed_time(b) for (k, a, b) in blk if k == "fwd"]
        b_ms = [a.elapsed_time(b) for (k, a, b) in blk if k == "bwd"]
        if f_ms and b_ms:
            blk_flops = 34.825e9 * B                                  # BASELINE.md §2: one ViP block fwd, per sample
            f_avg, b_avg = sum(f_ms) / len(f_ms), sum(b_ms) / len(b_ms)
            pk = measured_peaks()["tflops"]
            vit_block = {"what": f"one fused ViP encoder block (K3-K8), batch {B}, 2356 tokens, mean of {len(f_ms)} blocks",
                         "fwd_ms": round(f_avg, 3), "fwd_tflops": round(blk_flops / f_avg / 1e9, 1),
                         "fwd_frac_of_peak": round(blk_flops / f_avg / 1e9 / pk, 4),
                         "fwd_bwd_ms": round(f_avg + b_avg, 3),
                         "fwd_bwd_tflops": round(3 * blk_flops / (f_avg + b_avg) / 1e9, 1),
                         "fwd_bwd_frac_of_peak": round(3 * blk_flops / (f_avg + b_avg) / 1e9 / pk, 4), "peak_tflops": pk}

    model.clipmodel.overlap_text_tower = model.clipmodel.overlap_colsum = True
    # ---- extra (not part of `value`): the fused clip + AdamW step on this model's gradients (SURVEY.md §8f.1);
    #      HBM-bound: 28 B per parameter (read p, g, m, v; write p, m, v) + 4 B for the norm pass
    opt_info = None
    if world == 1:
        from xpretrain_b200.optimization.adamw import AdamW, build_e2e_optimizer_w_lr_mul
        opt = AdamW(build_e2e_optimizer_w_lr_mul(list(model.named_parameters()), 0.0, 0.2), lr=0.0, betas=(0.9, 0.98))
        step(*resident[0])                      # fresh gradients; lr = 0 keeps the weights (and later legs) unchanged
        for _ in range(2):
            opt.step(max_grad_norm=5.0)
        torch.cuda.synchronize()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for _ in range(5):
            opt.step(max_grad_norm=5.0)
        o1.record()
        torch.cuda.synchronize()
        n_par = sum(p.numel() for p in params)
        o_ms = o0.elapsed_time(o1) / 5
        hbm = measured_peaks().get("hbm_gbs", 6576.4)
        # a complete training step: fwd (incl. the per-forward fp32 -> bf16 weight re-cast) + gather + loss + bwd + clip + AdamW
        for _ in range(2):
            step(*resident[0]); opt.step(max_grad_norm=5.0)
        torch.cuda.synchronize()
        o2, o3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o2.record()
        for i in range(4):
            step(*resident[i % n_host]); opt.step(max_grad_norm=5.0)
        o3.record()
        torch.cuda.synchronize()
        t_ms = o2.elapsed_time(o3) / 4
        opt_info = {"what": "global-norm clip + AdamW over all parameters, 3 kernel launches", "ms": round(o_ms, 3),
                    "params": n_par, "gbs": round(32.0 * n_par / o_ms / 1e6, 1), "hbm_peak_gbs": hbm,
                    "frac_of_hbm_peak": round(32.0 * n_par / o_ms / 1e6 / hbm, 3),
                    "train_step": {"what": "fwd + gather + InfoNCE + bwd + clip + AdamW (lr 0), inputs resident",
                                   "ms": round(t_ms, 3), "pairs_per_s": round(B / t_ms * 1e3, 2)}}
        del opt

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    fm = flop_model()
    pairs = B * world
    value = pairs / (ms_resident * 1e-3)
    e2e_value = pairs / (ms_e2e * 1e-3)
    peaks = measured_peaks()
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_resident, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"CLIP-ViP ViT-B/16, {T} frames x 224^2, {Lt} tok, batch {B}/GPU (BASELINE.json configs[1]"
                               f"{'/[2]' if world > 1 else ''}); step = fwd + gather + InfoNCE + bwd"
                               f"{' + DP grad all-reduce' if world > 1 else ''}",
                   "global_batch": pairs, "frames": T, "tokens": Lt, "parallelism": f"dp{world}",
                   "sm_reserve_for_nccl": reserve, "grad_allreduce_dtype": os.environ.get("XP_GRAD_COMM", "fp32") if world > 1 else None,
                   "l2": "inputs (462 MB video + 40 GB activations per step) far exceed the 126 MB L2",
                   "weights": "random init with the reference's init statistics, fp32 masters, bf16 compute copies"},
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "ms_per_step": round(ms_e2e, 3),
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "last_loss": last["loss"]},
        "e2e_uint8_frames": e2e_u8,
        "gpu_launches": int(launches * world),
        "clocks": clocks,
        "roofline": roof,
        "vit_block": vit_block,
        "optimizer_step": opt_info,
        "whole_step": {"flops_per_pair": fm["train"], "tflops_per_gpu": round(value / world * fm["train"] / 1e12, 1),
                       "frac_of_peak": round(value / world * fm["train"] / 1e12 / peaks["tflops"], 4)},
    }
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(steps=CPU_MIN_STEPS, warmup=1, batch=CPU_BATCH)
        if not args.no_eager:
            del model, resident, slots
            torch.cuda.empty_cache()
            line["gpu_eager_baseline"] = gpu_eager_baseline(dev, B)
            if "value" in line["gpu_eager_baseline"]:
                line["gpu_eager_baseline"]["ours_over_eager_e2e"] = round(e2e_value / line["gpu_eager_baseline"]["value"], 2)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def ncu_traffic():
    """(dram__bytes_read + dram__bytes_write of one captured GEMM launch, what that launch was) from the committed ncu capture
    profiles/r02_ncu_gemm_traffic.json (a property of that capture, not of this run); (None, None) when none is committed."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_ncu_gemm_traffic.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return d["traffic_bytes"], {"algorithmic_bytes": d["algorithmic_bytes"]["total"],
                                    "launch": f"{d['kernel']} M={d['shape']['M']} N={d['shape']['N']} K={d['shape']['K']}",
                                    "source": "profiles/r02_ncu_gemm_traffic.json (one ncu --set full capture of this kernel, not of this run)"}
    except (OSError, KeyError, ValueError):
        return None, None


# -------------------------------------------------------------------------------- reference / CPU arm
def cpu_step_fn(batch):
    """The reference algorithm (oracle port of CLIP_ViP.py + loss.py) on the host: fwd + loss + bwd, fp32 eager."""
    import torch
    from oracle import clipvip_oracle as O
    cfg = O.ClipVipCfg()
    sd = O.init_state_dict(cfg, seed=0)
    sd = {k: (v.requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    video, ids, mask = O.synthetic_batch(batch, T_FRAMES, L_TOK, cfg, seed=1234)

    def fn():
        for v in sd.values():
            if v.is_floating_point():
                v.grad = None
        out = O.clip_vip_forward(sd, video, ids, mask, cfg)
        loss = O.nce_learnable_temp_loss(out["vis_features"], out["text_features"], sd["logit_scale"])
        loss.backward()
        return float(loss.detach())
    return fn


CPU_BATCH, CPU_THREADS_MAX, CPU_MIN_STEPS = 2, 32, 3


def cpu_threads():
    return min(os.cpu_count() or 1, CPU_THREADS_MAX)


def cpu_baseline(steps, warmup, batch=CPU_BATCH):
    """The reference algorithm on the host: FIXED batch and thread count, median of `steps` timed steps, identical in the
    in-line `cpu_baseline` object and in `--impl reference` (VERDICT r1: the one-step probe made the denominator swing 5x)."""
    import torch
    cores = os.cpu_count() or 1
    threads = cpu_threads()
    torch.set_num_threads(threads)
    fn = cpu_step_fn(batch)
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    dt = statistics.median(times)
    return {"value": round(batch / dt, 3), "unit": UNIT, "cores": threads, "host_cores": cores, "kind": "port",
            "sample": f"median of {len(times)} steps of batch {batch} x {T_FRAMES} frames x 224^2 + {L_TOK} tok, 12+12 layers, fp32 "
                      f"eager fwd+loss+bwd on {threads} threads (oracle/clipvip_oracle.py, pinned to the reference by "
                      f"tests/golden/make_golden.py)",
            "seconds_per_step": round(dt, 3), "seconds_min_max": [round(min(times), 3), round(max(times), 3)]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload != "clipvip":
        return run_reference_encoder(args)
    base = cpu_baseline(steps=args.steps, warmup=args.warmup, batch=CPU_BATCH)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(base["seconds_per_step"] * 1e3, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"CLIP-ViP ViT-B/16, {T_FRAMES} frames x 224^2, {L_TOK} tok; each step a bounded sample "
                                   f"of batch {CPU_BATCH} on the host CPU (the reference is pure PyTorch; its own "
                                   f"CPU path = fp32 eager); value = median step", "global_batch": CPU_BATCH,
                       "parallelism": "cpu", "timed_steps": args.steps},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(dev, batch):
    """north_star's 1-GPU bar, measured by the same run: the reference algorithm (oracle port: the same torch ops in the same
    order as CLIP_ViP.py / loss.py) in PyTorch eager on THIS B200 under bf16 autocast (`.to(bf16)` crashes in the reference,
    SURVEY.md §8c), fwd + InfoNCE + bwd, 2 warm-up + 3 timed steps; falls back to a smaller batch when eager runs out of memory."""
    import torch
    from oracle import clipvip_oracle as O
    cfg = O.ClipVipCfg()
    for B in (batch, batch // 2, batch // 4):
        if B < 1:
            break
        try:
            sd = {k: (v.to(dev).requires_grad_(True) if v.is_floating_point() else v.to(dev))
                  for k, v in O.init_state_dict(cfg, seed=0).items()}
            video, ids, mask = (t.to(dev) for t in O.synthetic_batch(B, T_FRAMES, L_TOK, cfg, seed=1234))

            def step():
                for v in sd.values():
                    if v.is_floating_point():
                        v.grad = None
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    out = O.clip_vip_forward(sd, video, ids, mask, cfg)
                    loss = O.nce_learnable_temp_loss(out["vis_features"].float(), out["text_features"].float(), sd["logit_scale"])
                loss.backward()

            for _ in range(2):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 3
            return {"what": "reference algorithm (oracle port), PyTorch eager, bf16 autocast, same GPU, same workload",
                    "batch": B, "ms_per_step": round(ms, 2), "value": round(B / ms * 1e3, 2), "unit": UNIT,
                    "max_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1)}
        except torch.OutOfMemoryError:
            sd = video = None
            torch.cuda.empty_cache()
    return {"what": "reference algorithm in PyTorch eager", "error": "out of memory at every batch tried"}


# ------------------------------------------------------- configs[3] / configs[4]: the video encoders of HD-VILA / LF-VILA
ENCODERS = {
    "timesformer": dict(
        metric="video clips/sec, HD-VILA TimeSformer (depth 4, dim 1024, 16 heads) fwd+bwd", unit="clips/s", batch=16,
        shape="[16, 8, 1024, 7, 7] = BASELINE.json configs[3]: 8 frames x 448^2 -> 7x7 feature grid (both table interpolations), "
              "batch 16/GPU"),
    "swin3d": dict(
        metric="videos/sec, LF-VILA Swin-3D video encoder (released VideoEncoder config) fwd+bwd", unit="videos/s", batch=8,
        shape="[8, 3, 32, 224, 224] = BASELINE.json configs[4]: 32 frames x 224^2, batch 8/GPU"),
}


def _encoder_flops(kind):
    """FLOP accounting only (BASELINE.md §2), read after the timed region."""
    if kind == "timesformer":
        from oracle import timesformer_oracle as TO
        return TO.flops_per_sample(TO.TimeSformerCfg(), 8, 7, 7)
    from oracle import swin3d_oracle as SO
    return SO.flops_per_sample(SO.Swin3DCfg(), 32, 224, 224)


def _encoder_ours(kind, dev, batch, seed):
    """(module with its own random init, pinned host input, weighted-sum target, forward) — nothing from oracle/ here."""
    import torch
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(0)
    if kind == "timesformer":
        from xpretrain_b200.modeling.timesformer import TimeSformer
        model = TimeSformer(depth=4, num_frames=7, H=10, W=16, embed_dim=1024, num_heads=16, drop_path_rate=0.0).to(dev).train()
        x = torch.randn(batch, 8, 1024, 7, 7, generator=g)
        fwd = lambda m, xin: m(xin)                                              # noqa: E731
    else:
        from xpretrain_b200.modeling.swin3d import SwinTransformer3D
        model = SwinTransformer3D(patch_norm=True, local_window=8, drop_path_rate=0.0).to(dev).train()
        x = torch.randn(batch, 3, 32, 224, 224, generator=g)
        fwd = lambda m, xin: m(xin)[0]                                           # noqa: E731
    with torch.no_grad():
        oshape = fwd(model, x[:1].to(dev)).shape
    n_out = 1
    for v in oshape[1:]:
        n_out *= v
    w_out = torch.randn((batch,) + tuple(oshape[1:]), generator=g) / float(n_out) ** 0.5
    return model, x, w_out, fwd


def _encoder_oracle(kind, batch, seed):
    import torch
    g = torch.Generator().manual_seed(7)
    if kind == "timesformer":
        from oracle import timesformer_oracle as TO
        cfg = TO.TimeSformerCfg()
        sd = TO.init_state_dict(cfg, seed=0)
        x = TO.synthetic_input(batch, 8, 7, 7, cfg, seed=seed)
        w_out = torch.randn(batch, 8, cfg.embed_dim, 7, 7, generator=g) / (batch * 8 * 49) ** 0.5
        return sd, x, w_out, (lambda sdo, xin: TO.timesformer_forward(sdo, xin, cfg))
    from oracle import swin3d_oracle as SO
    cfg = SO.Swin3DCfg()
    sd = SO.init_state_dict(cfg, seed=0)
    x = SO.synthetic_video(batch, 32, 224, 224, cfg, seed=seed)
    oshape = (batch, 32, 4, 4, 1024)          # 224 / 8 = 28 -> 14 -> 7 -> 4 (odd sizes are zero-padded by PatchMerging, :283-305)
    w_out = torch.randn(oshape, generator=g) / (32 * 4 * 4 * 1024) ** 0.5
    return sd, x, w_out, (lambda sdo, xin: SO.swin3d_forward(sdo, xin, cfg))


def encoder_cpu_baseline(kind, steps, warmup):
    """The reference encoder algorithm (oracle port, pinned bit-exact to the reference class by tests/golden/make_golden_*.py)
    on the host cores: fwd + bwd of a bounded sample (timesformer: 2 clips; swin3d: 1 video), median of `steps` steps."""
    import torch
    batch = 2 if kind == "timesformer" else 1
    threads = cpu_threads()
    torch.set_num_threads(threads)
    sd, x, w_out, oracle_fwd = _encoder_oracle(kind, batch, seed=1)
    sdo = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}

    def fn():
        for v in sdo.values():
            if v.is_floating_point():
                v.grad = None
        (oracle_fwd(sdo, x) * w_out).sum().backward()

    for _ in range(warmup):
        fn()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    dt = statistics.median(times)
    return {"value": round(batch / dt, 3), "unit": ENCODERS[kind]["unit"], "cores": threads, "host_cores": os.cpu_count() or 1,
            "kind": "port", "seconds_per_step": round(dt, 3),
            "sample": f"median of {len(times)} steps of batch {batch}, fp32 eager fwd+bwd of the oracle port on {threads} threads"}


def run_reference_encoder(args):
    kind = args.workload
    base = encoder_cpu_baseline(kind, steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": ENCODERS[kind]["metric"], "value": base["value"], "unit": base["unit"],
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(base["seconds_per_step"] * 1e3, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": ENCODERS[kind]["shape"] + "; each step a bounded CPU sample", "parallelism": "cpu"},
            "cpu_baseline": base, "e2e": {"value": base["value"], "unit": base["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_encoder(args):
    """`--workload timesformer|swin3d`: the same JSON contract for BASELINE.json configs[3] / configs[4] (VERDICT r1 item 6)."""
    import torch
    import torch.distributed as dist
    from xpretrain_b200 import ops
    from xpretrain_b200.utils import distributed as xdist

    kind = args.workload
    rank, local, world = xdist.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B = ENCODERS[kind]["batch"] if args.batch == PER_GPU_BATCH else args.batch
    model, x_host, w_out, fwd = _encoder_ours(kind, dev, B, seed=1 + rank)
    params = list(model.parameters())
    x_host = x_host.pin_memory()
    x_dev, w_out = x_host.to(dev), w_out.to(dev)

    last_step = {}

    def step(xin):
        for p in params:
            p.grad = None
        y = fwd(model, xin)
        loss = (y * w_out).sum()
        loss.backward()
        if world > 1:       # independent samples: data-parallel replicas, gradients averaged (hvd.DistributedOptimizer semantics)
            xdist.average_gradients(params)
        last_step.update(loss=loss.detach(), out=y.detach())
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    for _ in range(args.warmup):
        step(x_dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.reset_launch_count()
    ms_res = timed(lambda i: step(x_dev), args.steps)
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": last_step["loss"], "output": last_step["out"], "param_grads": flat_grads(params)})
    last = {}

    def e2e_step(i):
        xin = x_host.to(dev, non_blocking=True)
        last["loss"] = step(xin).detach().item()

    e2e_step(0)
    ms_e2e = timed(e2e_step, args.steps)
    rec = []
    ops.set_gemm_timer(rec)
    step(x_dev)
    torch.cuda.synchronize()
    ops.set_gemm_timer(None)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    g_ms = sum(a.elapsed_time(b) for (_, a, b) in rec)
    g_fl = sum(f for (f, _, _) in rec)
    peaks = measured_peaks()
    flops = _encoder_flops(kind)
    ach = g_fl / (g_ms * 1e-3) / 1e12
    value, e2e_value = B * world / (ms_res * 1e-3), B * world / (ms_e2e * 1e-3)
    line = {"metric": ENCODERS[kind]["metric"], "value": round(value, 2), "unit": ENCODERS[kind]["unit"], "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_res, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ENCODERS[kind]["shape"] + "; step = fwd + weighted-sum loss + bwd"
                                   + (" + DP gradient all-reduce" if world > 1 else ""),
                       "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2": "activations per step far exceed the 126 MB L2", "weights": "random init (reference statistics)"},
            "e2e": {"value": round(e2e_value, 2), "unit": ENCODERS[kind]["unit"], "ms_per_step": round(ms_e2e, 3),
                    "h2d_bytes_per_step": x_host.numel() * x_host.element_size(), "d2h_bytes_per_step": 4,
                    "last_loss": last.get("loss")},
            "gpu_launches": int(launches * world), "clocks": clocks,
            "roofline": {"kernel": "xp::gemm_kernel (tcgen05 bf16, all launches of one step)", "bound": "tensor",
                         "achieved": round(ach, 1), "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": round(ach / peaks["tflops"], 4),
                         "traffic": None, "peak_source": peaks["source"], "launches_per_step": len(rec),
                         "gemm_ms_per_step": round(g_ms, 3), "gemm_share_of_step": round(g_ms / ms_res, 4)},
            "whole_step": {"flops_per_sample": 3.0 * flops, "tflops_per_gpu": round(value / world * 3.0 * flops / 1e12, 1),
                           "frac_of_peak": round(value / world * 3.0 * flops / 1e12 / peaks["tflops"], 4)}}
    if world == 1:
        line["cpu_baseline"] = encoder_cpu_baseline(kind, steps=CPU_MIN_STEPS, warmup=1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="per-GPU batch (BASELINE.json configs[1]: 64)")
    ap.add_argument("--workload", default="clipvip", choices=["clipvip", "timesformer", "swin3d"],
                    help="clipvip = BASELINE.json configs[1]/[2] (default, the headline); timesformer = configs[3] (HD-VILA "
                         "spatio-temporal encoder); swin3d = configs[4] (LF-VILA Swin-3D video encoder)")
    ap.add_argument("--no-eager", action="store_true", help="skip the gpu_eager_baseline leg (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, features or encoder output, a fixed sample of the "
                         "parameter gradients) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "clipvip":
        run_ours(args)
    else:
        run_encoder(args)


if __name__ == "__main__":
    main()
