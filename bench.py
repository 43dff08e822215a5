#!/usr/bin/env python
"""Headline benchmark of the GDR-Net hot path (BASELINE.json configs[1]: ResNet-34 GDR-Net full fwd+bwd, batch 64 per GPU,
256x256 synthetic crops, losses included), one process per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm on the host cores (CPU oracle), same metric
    python bench.py --steps 20 --warmup 5 --dump-outputs DIR   # also write the last timed step's outputs to DIR/<name>.npy

One JSON line on stdout (rank 0).  `value` = crops/s of the whole job with inputs resident in HBM (device-timed, max over
ranks) in the PARITY-BACKED mode ("mixed": fp32-faithful 3-pass forward + single-pass fp16 backward; its B = 64 outputs are
checked against the CPU oracle at 1e-3 inside this run, key `parity_b64`); `e2e` = the same through the public module API
with pinned host inputs (H2D copies + D2H loss read in the timed region); `modes` = the other precision modes on the same
workload ("half" single-pass throughput mode, "fp32x3" 3-pass forward AND backward); `roofline` = tensor-core fraction of the
tcgen05 conv kernel family measured live with CUDA events; `cpu_baseline` = the CPU oracle timed on this box's host cores;
`cudnn_same_gpu` = the reference algorithm as PyTorch/cuDNN ops on this same GPU (TF32, channels_last, AMP variants).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "crops/sec (fwd+bwd, 256x256, bs64 per GPU)"
FWD_BWD_GFLOP_PER_CROP = 68.16  # SURVEY.md 8(d): 34.08 GMAC of Conv/ConvT/Linear, x2
FWD_GFLOP_PER_CROP = 22.823  # SURVEY.md 8(d): 11.4115 GMAC forward
BATCH_PER_GPU = 64
HEADLINE_MODE = os.environ.get("GDRN_BENCH_MODE", "mixed")  # the mode `value` / `e2e` are measured in


def finish_distributed(world):
    """End of a multi-rank run: one last barrier, then leave WITHOUT tearing the process group down.  The step graphs hold
    captured NCCL kernels; destroy_process_group() with them alive was observed to hang the ranks after the result line had
    been printed (r2, N=2), which would turn a finished run into a driver-side timeout.  A watchdog ends the process even if
    the barrier itself stalls."""
    sys.stdout.flush()
    if world <= 1:
        return
    import torch.distributed as dist

    threading.Timer(45.0, lambda: os._exit(0)).start()
    try:
        dist.barrier()
        torch.cuda.synchronize()
    except Exception:
        pass
    sys.stdout.flush()
    os._exit(0)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_sustained=d.get("bf16_tflops_sustained", 1453.0), bf16_burst=d.get("bf16_tflops", 1718.7),
                    hbm=d.get("hbm_gbs", 6571.6), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


WITH_SYM = False  # "ycbv" for --config ycbv (BASELINE.json configs[4]): PM_LOSS_SYM with a 21-object symmetry set


def build(precision: str, device: str = "cuda"):
    from gdr_net_b200 import GDRN as G
    from gdr_net_b200 import synth
    from gdr_net_b200.config import a6_config

    cfg = a6_config(device=device, pm_loss_sym=bool(WITH_SYM))
    model, opt = G.build_model_optimizer(cfg, precision=precision)
    # seeded Kaiming-scale weights (SURVEY P1: the reference's std=1e-3 init is degenerate without ImageNet weights)
    sd = synth.seeded_state_dict(model.state_dict(), seed=0)
    model.load_state_dict(sd)
    model.train()
    return model, opt


def device_batch(batch, dev):
    return {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in batch.items()}


def aux_from_batch(b):
    return dict(roi_coord_2d=b["roi_coord_2d"], roi_cams=b["roi_cam"], roi_centers=b["roi_center"], roi_whs=b["roi_wh"],
                roi_extents=b["roi_extent"], resize_ratios=b["resize_ratio"], gt_xyz=b["roi_xyz"],
                gt_mask_trunc=b["roi_mask_trunc"], gt_mask_visib=b["roi_mask_visib"], gt_region=b["roi_region"],
                gt_ego_rot=b["ego_rot"], gt_points=b["roi_points"], sym_infos=b.get("sym_info"), gt_trans=b["trans"],
                gt_trans_ratio=b["roi_trans_ratio"])


DUMP_HEAD_ROWS = 1 << 16   # of the B*64*64 head pixels (69 channels each)
DUMP_GRAD_ELEMS = 1 << 21  # of the ~35M entries of the flat gradient
DUMP_MAX_BYTES = 64 << 20


def train_step_outputs(last, flat_grad):
    """What a train step hands its caller, as host arrays for --dump-outputs: the 8 losses (engine.LOSS_NAMES order), the decoded
    poses, and a fixed sample (seed 0, same rows / entries every run) of the 69-channel head maps and of the flat gradient, with
    the sampled row / entry indices.  The full head and gradient (~210 MB) are sampled to stay under 64 MB."""
    g = torch.Generator().manual_seed(0)
    head = last["logits"].reshape(-1, 72)[:, :69]  # NHWC pixel rows: row = crop * 4096 + y * 64 + x
    rows = torch.randperm(head.shape[0], generator=g)[:DUMP_HEAD_ROWS].sort().values
    idx = torch.randperm(flat_grad.numel(), generator=g)[:DUMP_GRAD_ELEMS].sort().values
    f32 = lambda t: t.detach().float().cpu().numpy()  # noqa: E731
    return {"losses": f32(last["losses"]), "rot": f32(last["rot"]), "trans": f32(last["trans"]),
            "head_sample": f32(head[rows.to(head.device)]), "head_sample_rows": rows.double().numpy(),
            "grad_sample": f32(flat_grad[idx.to(flat_grad.device)]), "grad_sample_index": idx.double().numpy()}


def dump_outputs(out_dir, arrays):
    """DIR/<name>.npy per array (float32 / float64 only)."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    global BATCH_PER_GPU, WITH_SYM, METRIC
    if args.config == "ycbv":
        BATCH_PER_GPU, WITH_SYM = 32, "ycbv"
        METRIC = "crops/sec (fwd+bwd, 256x256, bs32 per GPU, YCB-V symmetric PM loss)"
    from gdr_net_b200 import synth
    from gdr_net_b200.capi import launch_count
    from gdr_net_b200.dist import GradAllReducer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    B = BATCH_PER_GPU
    peaks = load_peaks()
    # --dump-outputs: the train steps use the engine's ordered two-stage reductions for the BatchNorm statistics and backward
    # sums instead of fp32 atomics, so that with the same arguments a step computes the same outputs every run and two builds
    # can be compared output for output (the atomics' ordering jitter, ~1e-7, is amplified by the network's ReLU / max-pool
    # decisions to ~1e-4 in the head maps and ~2e-2 in the gradients).  It costs one extra read of every pre-BN tensor in
    # forward, so without --dump-outputs the default (atomics) path is timed; the JSON records which one ran.
    deterministic = args.dump_outputs is not None

    def one_mode(precision, steps, warmup, with_clocks, capture_outputs=False):
        model, _opt = build(precision)
        eng = model.engine
        eng.deterministic = deterministic
        reducer = GradAllReducer(eng.flat_grad, eng.named_params) if world > 1 else None
        eng.grad_hook = reducer
        batch = device_batch(synth.make_batch(B, seed=100 + rank, with_sym=WITH_SYM), dev)
        x = batch["roi_img"].float().contiguous()
        aux = {k: (v.float().contiguous() if isinstance(v, torch.Tensor) and v.dtype != torch.long else v)
               for k, v in aux_from_batch(batch).items()}
        gl = torch.ones(8, device=dev)
        last = {}

        def eager_step():
            res = eng.forward(x, aux, train_bn=True, do_loss=True)
            eng.backward(gl)
            if reducer is not None:
                reducer.finish()
            last.update(losses=res["losses"], logits=res["logits"], rot=res["rot"], trans=res["trans"])
            return res["losses"]

        step = eager_step
        graphed = None
        if args.graph:
            from gdr_net_b200.engine import GraphedTrainStep

            # forward + losses + backward + (N > 1) the bucketed NCCL all-reduces on their side stream: ONE graph per step
            graphed = GraphedTrainStep(eng, x, aux, train_bn=True)
            step = graphed
            last.update(losses=graphed.losses, logits=graphed.logits, rot=graphed.rot, trans=graphed.trans)

        for _ in range(warmup):
            losses = step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local) if (with_clocks and rank == 0) else None  # one poller per job, not per rank
        if sampler:
            sampler.start()
        l0 = launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        profiling = os.environ.get("GDRN_PROFILE") == "1"  # ncu --profile-from-start off: capture the timed steps only
        if profiling:
            torch.cuda.profiler.start()
        e0.record()
        for _ in range(steps):
            losses = step()
        e1.record()
        torch.cuda.synchronize()
        if profiling:
            torch.cuda.profiler.stop()
        ms = e0.elapsed_time(e1) / steps
        launches = (launch_count() - l0) // steps
        clocks = sampler.stop() if sampler else None
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(t)
        assert torch.isfinite(losses).all(), "non-finite losses"
        step_losses, step_logits = last["losses"].clone(), last["logits"].clone()  # outputs of the last TIMED step
        # taken before the launch-count step below, which recomputes the same buffers
        outputs = train_step_outputs(last, eng.flat_grad) if capture_outputs else None
        if graphed is not None:  # launches inside a replayed graph are not seen by the library's host-side counter
            l1 = launch_count()
            eager_step()
            launches = launch_count() - l1
            torch.cuda.synchronize()
        return dict(model=model, eng=eng, ms=ms, launches=launches, clocks=clocks, batch=batch, losses=step_losses,
                    logits=step_logits, graphed=graphed is not None, precision=precision, outputs=outputs)

    main = one_mode(HEADLINE_MODE, args.steps, args.warmup, with_clocks=True, capture_outputs=bool(args.dump_outputs) and rank == 0)
    if main["outputs"] is not None:
        dump_outputs(args.dump_outputs, main.pop("outputs"))
    ms = main["ms"]
    value = world * B / (ms / 1e3)
    mode_desc = {
        "mixed": "fp32-faithful forward (hi/lo fp16 planes = 22-bit operands, 3 tcgen05 passes, fp32 accumulate) + single-pass "
                 "fp16 backward (loss scale 1024); forward outputs / losses checked at 1e-3 against the CPU oracle at B=64 "
                 "(parity_b64), gradients at the fp32x3 bound (tests/test_parity_b64_gpu.py)",
        "fp32x3": "hi/lo fp16 planes (22-bit operands), 3 tcgen05 passes in forward and backward",
        "half": "single fp16 plane, one tcgen05 pass (TF32-class operands; NOT inside the 1e-3 parity bound)",
    }

    out = {
        "metric": METRIC, "value": round(value, 1), "unit": "crops/s", "per_gpu": round(value / world, 1), "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": {"mixed": "fp16x3 fwd / fp16 bwd, f32 accumulate", "fp32x3": "fp16x3, f32 accumulate", "half": "fp16, f32 accumulate"}[HEADLINE_MODE],
        "data": "synthetic",
        "config": {"workload": ("configs[1]: ResNet-34 GDR-Net (a6_cPnP shapes) full fwd+bwd incl. all 8 losses, train-mode BN, "
                                "batch 64/GPU, 256x256 synthetic crops, seeded Kaiming weights") if not WITH_SYM else
                               ("configs[4]: YCB-V 21-object config (PM_LOSS_SYM: closest symmetric GT among up to 628 candidates per "
                                "crop, device-resident table), ResNet-34 GDR-Net full fwd+bwd incl. all 8 losses, batch 32/GPU, 256x256 synthetic crops"),
                   "precision_mode": HEADLINE_MODE + ": " + mode_desc[HEADLINE_MODE],
                   "global_batch": world * B, "parallelism": f"dp{world}",
                   "l2": "activations per step (>2 GB) exceed the 126 MB L2; no explicit flush",
                   "launch": "whole step (incl. the NCCL all-reduces at N>1) replayed as one CUDA graph" if main["graphed"] else "eager (one ctypes call per kernel)",
                   "grad_exchange": "bucketed NCCL all-reduce (AVG) of the flat 140 MB fp32 gradient buffer on a side stream, overlapped with backward, captured in the step graph" if world > 1 else "none",
                   "deterministic": deterministic},
        "clocks": main["clocks"], "gpu_launches": int(main["launches"]),
    }

    if args.quick:
        if rank == 0:
            print(json.dumps(out), flush=True)
        finish_distributed(world)
        return
    if rank == 0 or world > 1:
        # ---- e2e through the public module API with pinned host inputs (H2D + D2H inside the timed region)
        model = main["model"]
        model.engine.grad_hook = main["eng"].grad_hook
        model.use_cuda_graphs = args.graph  # forward / backward graphs (incl. the all-reduces) behind the public module API
        host = synth.make_batch(B, seed=200 + rank, with_sym=WITH_SYM)
        pinned = {k: (v.pin_memory() if isinstance(v, torch.Tensor) else v) for k, v in host.items()}
        h2d = sum(v.numel() * v.element_size() for v in pinned.values() if isinstance(v, torch.Tensor))
        reducer = main["eng"].grad_hook

        copy_stream = torch.cuda.Stream()

        def upload():
            """H2D copy of one step's inputs from pinned host memory on the copy stream (overlaps the previous step)."""
            with torch.cuda.stream(copy_stream):
                b = {k: (v.to(dev, non_blocking=True) if isinstance(v, torch.Tensor) else v) for k, v in pinned.items()}
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return b, ev

        loss_host = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
        read_back = []

        def e2e_step(cur, i):
            b, ev = cur
            nxt = upload()  # next step's inputs start moving while this step computes
            torch.cuda.current_stream().wait_event(ev)
            for t in b.values():
                if isinstance(t, torch.Tensor):
                    t.record_stream(torch.cuda.current_stream())
            for p in model.parameters():
                p.grad = None
            _, loss_dict = model(b["roi_img"], **synth.forward_kwargs(b, train=True))
            total = sum(loss_dict.values())
            total.backward()
            if reducer is not None:
                reducer.finish()
            # D2H read of the step's loss, software-pipelined like the H2D side: the 4-byte copy of step i is queued behind
            # its backward, and the host consumes step i-1's value (already landed in pinned memory) while step i runs.
            # Every step's loss is read inside the timed region (the last one by drain()); the GPU never waits for the host.
            loss_host[i & 1].copy_(total.detach(), non_blocking=True)
            loss_ev[i & 1].record()
            if i > 0:
                loss_ev[(i - 1) & 1].synchronize()
                read_back.append(float(loss_host[(i - 1) & 1]))
            return nxt

        def drain(i_last):
            loss_ev[i_last & 1].synchronize()
            read_back.append(float(loss_host[i_last & 1]))

        n_e2e = args.steps
        cur = upload()
        # >= 8 untimed steps: the first one captures the forward / backward graphs, the next few let the caching allocator reach
        # its steady state (the prefetched input tensors are held by record_stream for a step, so early steps still cudaMalloc)
        n_w = max(8, args.warmup)
        for i in range(n_w):
            cur = e2e_step(cur, i)
        drain(n_w - 1)
        torch.cuda.synchronize()
        # three timed regions of exactly K steps each, the MEDIAN is reported (all three are in `regions_ms`): a region is
        # 0.2 s long, so one host-side hiccup (GC pause, a page fault in the pinned staging) would otherwise move it by 10-20 %
        regions = []
        for rep in range(3):
            if world > 1:
                dist.barrier()
            read_back.clear()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_host0 = time.perf_counter()
            e0.record()
            for i in range(n_e2e):
                cur = e2e_step(cur, i)
            drain(n_e2e - 1)
            e1.record()
            torch.cuda.synchronize()
            t_host = (time.perf_counter() - t_host0) * 1e3 / n_e2e
            assert len(read_back) == n_e2e and all(v == v and abs(v) < 1e6 for v in read_back), read_back
            regions.append(max(e0.elapsed_time(e1) / n_e2e, t_host))  # device events and the host clock must agree
        ms_e2e = sorted(regions)[1]
        if world > 1:
            t = torch.tensor([ms_e2e], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e2e = float(t)
        out["e2e"] = {"value": round(world * B / (ms_e2e / 1e3), 1), "unit": "crops/s", "ms_per_step": round(ms_e2e, 3),
                      "steps": n_e2e, "regions_ms": [round(r, 3) for r in regions], "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                      "api": "gdr_net_b200.GDRN.GDRN.forward(...do_loss=True) + sum(loss_dict.values()).backward() (precision "
                             f"'{HEADLINE_MODE}'); every step's inputs are copied from pinned host memory (prefetched one step ahead "
                             "on a copy stream) and every step's loss is read back to the host (4-byte async D2H, consumed one step later)"}

    if rank == 0:
        # ---- roofline of the dominant kernel family (tcgen05 implicit-GEMM conv: fwd + dgrad + wgrad), measured live
        out["roofline"] = roofline_live(main, peaks)
        if world == 1:
            main_small = dict(losses=main["losses"].cpu(), logits=main["logits"].cpu(), precision=main["precision"])
            del main["model"], main["eng"], main["logits"]
            torch.cuda.empty_cache()
            out["modes"] = {}
            for prec in ("half", "fp32x3", "mixed"):
                if prec == HEADLINE_MODE:
                    out["modes"][prec] = {"value": round(B / (ms / 1e3), 1), "unit": "crops/s", "ms_per_step": round(ms, 3), "headline": True}
                    continue
                try:
                    r = one_mode(prec, args.steps, 3, with_clocks=False)
                    out["modes"][prec] = {"value": round(B / (r["ms"] / 1e3), 1), "unit": "crops/s", "ms_per_step": round(r["ms"], 3),
                                          "what": mode_desc[prec]}
                    del r
                    torch.cuda.empty_cache()
                except Exception as e:  # pragma: no cover
                    out["modes"][prec] = {"error": str(e)[:200]}
            try:
                out["inference"] = inference_bench(B, dev, peaks)
            except Exception as e:  # pragma: no cover
                out["inference"] = {"error": str(e)[:300]}
            cb, parity = cpu_baseline(sample_batch=args.cpu_batch, iters=args.cpu_iters, check=main_small)
            out["cpu_baseline"] = cb
            out["parity_b64"] = parity
            try:
                out["cudnn_same_gpu"] = cudnn_same_gpu(B, dev)
            except Exception as e:  # pragma: no cover
                out["cudnn_same_gpu"] = {"error": str(e)[:300]}
        print(json.dumps(out), flush=True)
    finish_distributed(world)


def roofline_live(main, peaks):
    """Time every tcgen05 GEMM launch of one step with CUDA events (on the launching stream) and divide the
    algorithmic FLOPs (2*M*N*K of the convolution / linear it implements) by the summed durations."""
    from gdr_net_b200 import ops

    eng = main["eng"]
    hook, eng.grad_hook = eng.grad_hook, None  # rank-0-only instrumentation pass: no collectives
    side, eng.wgrad_side_stream = eng.wgrad_side_stream, False  # the per-launch CUDA events bracket kernels on ONE stream
    batch = main["batch"]
    x = batch["roi_img"].float().contiguous()
    aux = {k: (v.float().contiguous() if isinstance(v, torch.Tensor) and v.dtype != torch.long else v)
           for k, v in aux_from_batch(batch).items()}
    records = []
    orig = {n: getattr(ops, n) for n in ("conv_fwd", "gemm_fwd", "conv_dgrad_s2", "conv_wgrad", "gemm_wgrad")}

    from gdr_net_b200.capi import C as _C

    def timed(name, fn, flops_of):
        def wrapper(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            variant = _C.load().gdrn_last_gemm_variant() if name in ("conv_fwd", "gemm_fwd", "conv_dgrad_s2") else 0
            passes = a[1].nsplit if name in ("conv_wgrad", "gemm_wgrad") else a[0].nsplit  # tcgen05 passes per algorithmic MAC
            records.append((name, flops_of(*a, **k), e0, e1, variant, passes))
            return r

        return wrapper

    def f_conv(x_, wp, Cout, KH, KW, stride, pad, **k):
        N, H, W, Cin = x_.shape
        return 2.0 * N * (H // stride) * (W // stride) * Cout * Cin * KH * KW * k.get("algo_scale", 1.0)

    def f_dg2(du, wd, Cx, K, pad, **k):  # stride-2 dgrad by output-parity phases: exactly the conv's MACs
        N, Ho, Wo, Cy = du.shape
        return 2.0 * N * Ho * Wo * Cy * Cx * K * K

    def f_gemm(a, wp, N, **k):
        return 2.0 * a.shape[0] * N * a.shape[1]

    def f_cw(dy, x_, ws, Cout, KH, KW, stride, pad, ksplit=0):
        N, H, W, Cin = x_.shape
        return 2.0 * N * (H // stride) * (W // stride) * Cout * Cin * KH * KW

    def f_gw(dy, x_, ws, ksplit=0):
        return 2.0 * dy.shape[0] * dy.shape[1] * x_.shape[1]

    ops.conv_fwd = timed("conv_fwd", orig["conv_fwd"], f_conv)
    ops.gemm_fwd = timed("gemm_fwd", orig["gemm_fwd"], f_gemm)
    ops.conv_dgrad_s2 = timed("conv_dgrad_s2", orig["conv_dgrad_s2"], f_dg2)
    ops.conv_wgrad = timed("conv_wgrad", orig["conv_wgrad"], f_cw)
    ops.gemm_wgrad = timed("gemm_wgrad", orig["gemm_wgrad"], f_gw)
    try:
        gl = torch.ones(8, device=x.device)
        e0, em, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        n_fwd = 0
        for it in range(3):
            records.clear()
            e0.record()
            eng.forward(x, aux, train_bn=True, do_loss=True)
            em.record()
            n_fwd = len(records)
            eng.backward(gl)
            e1.record()
        torch.cuda.synchronize()
    finally:
        for n, f in orig.items():
            setattr(ops, n, f)
        eng.grad_hook = hook
        eng.wgrad_side_stream = side
    step_ms, fwd_ms = e0.elapsed_time(e1), e0.elapsed_time(em)
    fam, inst = {}, {}
    fwd_fl = fwd_gemm_ms = fwd_mma = 0.0
    tot_mma = 0.0
    for i, (name, fl, a, b, variant, passes) in enumerate(records):
        ms_ = a.elapsed_time(b)
        d = fam.setdefault(name, [0.0, 0.0, 0, 0.0])
        d[0] += fl
        d[1] += ms_
        d[2] += 1
        d[3] += fl * passes
        tot_mma += fl * passes
        if i < n_fwd:
            fwd_fl += fl
            fwd_gemm_ms += ms_
            fwd_mma += fl * passes
        if variant:
            kname = "gemm_fwd2_kernel" if variant >= 10000 else "gemm_fwd_kernel"  # fwd2 = cta_group::2 pair tiles
            key = f"gdrn::{kname}<{(variant % 10000) // 10}, {variant % 10}>"
            d = inst.setdefault(key, [0.0, 0.0, 0, 0.0])
            d[0] += fl
            d[1] += ms_
            d[2] += 1
            d[3] += fl * passes
    tot_fl = sum(v[0] for v in fam.values())
    tot_ms = sum(v[1] for v in fam.values())
    # dominant kernel = the instantiation with the largest time share of the step
    dom = max(inst.items(), key=lambda kv: kv[1][1])
    dom_tflops = dom[1][0] / (dom[1][1] * 1e-3) / 1e12
    dom_mma = dom[1][3] / (dom[1][1] * 1e-3) / 1e12
    # the timed region of this benchmark is a fraction of a second at full boost clocks: the comparator is the BURST peak
    peak = peaks["bf16_burst"]
    prof = {}
    ppath = os.path.join(ROOT, "profiles", "ncu_kernel_facts.json")  # written from committed ncu captures, keyed by kernel name
    if os.path.exists(ppath):
        prof = json.load(open(ppath)).get(dom[0], {})
    tf = lambda fl, ms_: round(fl / (ms_ * 1e-3) / 1e12, 1) if ms_ > 0 else None  # noqa: E731
    return {
        "bound": "tensor", "kernel": dom[0] + " (tcgen05 implicit-GEMM conv forward / dgrad" + (", cta_group::2 pair tiles)" if "fwd2" in dom[0] else ")"),
        "achieved": round(dom_tflops, 1), "peak": peak, "unit": "TFLOP/s", "frac": round(dom_tflops / peak, 4),
        "peak_source": "bf16_tflops (burst; fp16 and bf16 tcgen05 rates are equal) of " + peaks["source"]
                       + ": the timed region is < 1 s at full boost clocks",
        "achieved_note": "ALGORITHMIC FLOPs (2*M*N*K of the conv) / summed launch durations; the 3-pass instantiations execute "
                         "3 tcgen05 MMAs per algorithmic MAC, `mma_tflops` is that executed rate (what the tensor pipe sees)",
        "mma_tflops": round(dom_mma, 1), "mma_frac": round(dom_mma / peak, 4),
        "launches_per_step": dom[1][2], "avg_launch_ms": round(dom[1][1] / dom[1][2], 4),
        "algorithmic_gflop_per_launch": round(dom[1][0] / dom[1][2] / 1e9, 2), "share_of_step": round(dom[1][1] / step_ms, 3),
        "traffic": prof.get("dram_bytes_per_launch"), "traffic_note": prof.get("note", "no ncu --set full capture of this instantiation committed yet"),
        "tensor_pipe_pct_ncu": prof.get("tensor_pipe_pct"),
        "gemm_family": {"achieved": tf(tot_fl, tot_ms), "frac": round(tot_fl / (tot_ms * 1e-3) / 1e12 / peak, 4),
                        "mma_tflops": tf(tot_mma, tot_ms), "mma_frac": round(tot_mma / (tot_ms * 1e-3) / 1e12 / peak, 4),
                        "share_of_step": round(tot_ms / step_ms, 3), "launches_per_step": sum(v[2] for v in fam.values()),
                        "algorithmic_gflop_per_step": round(tot_fl / 1e9, 1)},
        "forward_only": {"what": "backbone + head + Patch-PnP forward incl. losses (eager pass, CUDA events)",
                         "ms": round(fwd_ms, 3), "gemm_ms": round(fwd_gemm_ms, 3),
                         "algorithmic_tflops_gemm": tf(fwd_fl, fwd_gemm_ms), "mma_tflops_gemm": tf(fwd_mma, fwd_gemm_ms),
                         "mma_frac_gemm": round(fwd_mma / (fwd_gemm_ms * 1e-3) / 1e12 / peak, 4),
                         "algorithmic_tflops_wall": tf(FWD_GFLOP_PER_CROP * 1e9 * BATCH_PER_GPU, fwd_ms),
                         "mma_frac_wall": round(fwd_mma / (fwd_ms * 1e-3) / 1e12 / peak, 4)},
        "instantiations": {k: {"tflops": tf(v[0], v[1]), "mma_tflops": tf(v[3], v[1]), "ms": round(v[1], 3), "launches": v[2]}
                           for k, v in sorted(inst.items(), key=lambda kv: -kv[1][1])},
        "families": {k: {"tflops": tf(v[0], v[1]), "mma_tflops": tf(v[3], v[1]), "ms": round(v[1], 3), "launches": v[2]} for k, v in fam.items()},
        "whole_step_tflops": round(FWD_BWD_GFLOP_PER_CROP * BATCH_PER_GPU / main["ms"], 1),
        "whole_step_frac": round(FWD_BWD_GFLOP_PER_CROP * BATCH_PER_GPU / main["ms"] / peak, 4),
    }


def run_pnp(args):
    """BASELINE.json configs[3]: stand-alone Patch-PnP, [512, nIn, 64, 64] correspondence maps -> rot6d | t (inference)."""
    from gdr_net_b200 import synth
    from gdr_net_b200.capi import launch_count
    from gdr_net_b200.GDRN import ConvPnPNet
    from oracle import gdrn_oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    B, nin = 512, args.nin
    c_feat = nin - 64
    peaks = load_peaks()
    net = ConvPnPNet(nIn=nin).to(dev)
    sd = synth.seeded_state_dict({"pnp_net." + k: v for k, v in net.state_dict().items()}, seed=11)
    net.load_state_dict({k[len("pnp_net."):]: v for k, v in sd.items()})
    g = synth._gen(7 + rank, "pnp_bench")
    coor_h = torch.rand(B, c_feat, 64, 64, generator=g).pin_memory()
    reg_h = torch.softmax(2.0 * torch.randn(B, 64, 64, 64, generator=g), dim=1).pin_memory()
    ext_h = (0.05 + 0.25 * torch.rand(B, 3, generator=g)).pin_memory()
    coor, reg, ext = coor_h.to(dev), reg_h.to(dev), ext_h.to(dev)
    out = {}
    results = {}
    for precision in ("fp32x3", "half"):
        net.precision = precision
        for _ in range(max(3, args.warmup)):
            rot, t = net(coor, reg, ext)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local) if (rank == 0 and precision == "fp32x3") else None
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            rot, t = net(coor, reg, ext)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        rot, t = rot.cpu(), t.cpu()  # outputs of the last timed step (the graph's output buffers are reused below)
        clocks = sampler.stop() if sampler else None
        if world > 1:
            tt = torch.tensor([ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt)
        # e2e: host buffers in, host results out, every step
        e0.record()
        n_e2e = args.steps
        for _ in range(n_e2e):
            r_, t_ = net(coor_h.to(dev, non_blocking=True), reg_h.to(dev, non_blocking=True), ext_h.to(dev, non_blocking=True))
            r_host, t_host = r_.cpu(), t_.cpu()
        e1.record()
        torch.cuda.synchronize()
        ms_e2e = e0.elapsed_time(e1) / n_e2e
        if world > 1:
            tt = torch.tensor([ms_e2e], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms_e2e = float(tt)
        results[precision] = dict(ms=ms, ms_e2e=ms_e2e, rot=rot, t=t, clocks=clocks)
    if rank != 0:
        finish_distributed(world)
        return
    main = results["fp32x3"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rot": main["rot"].float().numpy(), "t": main["t"].float().numpy()})
    # algorithmic work (SURVEY 8d config 4): Conv / Linear MACs x 2 with the true nIn; bytes = fp32 input maps + fp32 weights
    flops = 2.0 * B * (1024 * 128 * 9 * nin + 256 * 128 * 9 * 128 + 64 * 128 * 9 * 128 + 8192 * 1024 + 1024 * 256 + 256 * 9)
    wbytes = 4.0 * sum(p.numel() for p in net.parameters())
    abytes = 4.0 * B * nin * 4096 + wbytes
    l0 = launch_count()
    net._runner.use_cuda_graphs = False
    net(coor, reg, ext)
    launches = launch_count() - l0
    net._runner.use_cuda_graphs = True
    # parity (the oracle as checker) + CPU baseline on a bounded sample
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    with torch.no_grad():
        t0 = time.perf_counter()
        rot_ref, t_ref = O.pnp_forward(coor_h, reg_h, ext_h, sd)
        t_cpu = time.perf_counter() - t0
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())  # noqa: E731
    parity = {p_: {"rot_rel_l2": float(f"{rel(results[p_]['rot'], rot_ref):.3e}"), "t_rel_l2": float(f"{rel(results[p_]['t'], t_ref):.3e}")} for p_ in results}
    assert parity["fp32x3"]["rot_rel_l2"] <= 1e-3 and parity["fp32x3"]["t_rel_l2"] <= 1e-3, parity
    # the reference nn.Conv2d / GroupNorm / Linear stack on this GPU (cuDNN, TF32 default, cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    sd_dev = {k: v.to(dev) for k, v in sd.items()}
    with torch.no_grad():
        for _ in range(3):
            O.pnp_forward(coor, reg, ext, sd_dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            O.pnp_forward(coor, reg, ext, sd_dev)
        e1.record()
        torch.cuda.synchronize()
    ms_cudnn = e0.elapsed_time(e1) / 10
    ms = main["ms"]
    line = {
        "metric": "crops/sec (stand-alone Patch-PnP forward, 64x64 maps, bs512 per GPU)", "value": round(world * B / ms * 1e3, 1), "unit": "crops/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp16x3, f32 accumulate", "data": "synthetic",
        "config": {"workload": f"configs[3]: Patch-PnP isolation, [512, {nin}, 64, 64] correspondence maps (xyz{'+2D' if c_feat == 5 else ''} + 64 region "
                               "channels) + extents -> rot6d | t; NCHW fp32 inputs resident in HBM; one CUDA graph per step "
                               "(pack -> 3x(conv3x3 s2 + GN + ReLU) -> fc1 -> fc2 -> fc_r|fc_t)",
                   "global_batch": world * B, "parallelism": f"replicas x{world}", "l2": "input maps (580 MB) exceed the 126 MB L2"},
        "clocks": main["clocks"], "gpu_launches": int(launches),
        "e2e": {"value": round(world * B / main["ms_e2e"] * 1e3, 1), "unit": "crops/s", "ms_per_step": round(main["ms_e2e"], 3),
                "h2d_bytes_per_step": int(coor_h.numel() * 4 + reg_h.numel() * 4 + ext_h.numel() * 4), "d2h_bytes_per_step": B * 9 * 4,
                "api": "ConvPnPNet.forward(coor_feat, region, extents) with pinned host tensors in, host rot/t out, every step"},
        "roofline": {"bound": "hbm", "achieved": round(abytes / (ms * 1e-3) / 1e9, 1), "peak": peaks["hbm"], "unit": "GB/s",
                     "frac": round(abytes / (ms * 1e-3) / 1e9 / peaks["hbm"], 4), "traffic": None,
                     "algorithmic_bytes_per_step": abytes,
                     "tensor_bound": {"achieved": round(flops / (ms * 1e-3) / 1e12, 1), "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                                      "frac": round(flops / (ms * 1e-3) / 1e12 / peaks["bf16_burst"], 4),
                                      "algorithmic_gflop_per_step": round(flops / 1e9, 1)},
                     "note": "the path sits at the ridge (SURVEY 8d: ~229 FLOP/B): both bounds reported; whole graph (7 GEMM + 4 HBM-bound launches), not one kernel"},
        "modes": {"half": {"value": round(world * B / results["half"]["ms"] * 1e3, 1), "unit": "crops/s", "ms_per_step": round(results["half"]["ms"], 4)}},
        "parity_b512": dict(parity, tolerance=1e-3, checker="oracle pnp_forward (conv_pnp_net.py:111-157 restated) on the same maps / weights"),
        "cpu_baseline": {"value": round(B / t_cpu, 1), "unit": "crops/s", "cores": cores, "kind": "port",
                         "sample": f"one forward of the {B}-crop batch, torch CPU fp32, {cores} threads"},
        "cudnn_same_gpu": {"value": round(B / ms_cudnn * 1e3, 1), "unit": "crops/s", "ms_per_step": round(ms_cudnn, 3),
                           "what": "the reference nn stack restated (F.conv2d / group_norm / linear, NCHW fp32, TF32 convs, cudnn.benchmark) on this GPU"},
    }
    print(json.dumps(line), flush=True)
    finish_distributed(world)


def inference_bench(B, dev, peaks, steps=20, warm=5):
    """Forward-only (eval mode, the reference's inference caller gdrn_evaluator.py:568-580) through the public module API with
    inputs resident: every conv + BatchNorm (+ identity) + ReLU is ONE kernel (BatchNorm folded into the packed weights and
    the GEMM epilogue).  Reports crops/s and the forward tensor-core utilisation (north_star: >= 60 % on backbone+head fwd)."""
    from gdr_net_b200 import synth

    batch = device_batch(synth.make_batch(B, seed=100), dev)
    kw = synth.forward_kwargs(batch, train=False)
    res = {}
    for precision, passes in (("mixed", 3), ("half", 1)):
        model, _ = build(precision)
        model.eval()
        model.use_cuda_graphs = True  # the inference forward is replayed as one CUDA graph
        with torch.no_grad():
            for _ in range(warm):
                out = model(batch["roi_img"], **kw)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = model(batch["roi_img"], **kw)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        assert torch.isfinite(out["rot"]).all() and torch.isfinite(out["trans"]).all()
        tf = FWD_GFLOP_PER_CROP * B / ms  # algorithmic TFLOP/s (GFLOP / ms)
        res[precision] = {"value": round(B / ms * 1e3, 1), "unit": "crops/s", "ms_per_step": round(ms, 3),
                          "algorithmic_tflops": round(tf, 1), "mma_tflops": round(tf * passes, 1),
                          "mma_frac_of_burst_peak": round(tf * passes / peaks["bf16_burst"], 4)}
        del model
        torch.cuda.empty_cache()
    res["what"] = ("GDRN.forward(do_loss=False) in eval mode, batch 64, use_cuda_graphs=True (one graph replay per forward), inputs resident; "
                   "folded conv+BN(+identity)+ReLU epilogues; 'mixed' = fp32-faithful 3-pass operands (1e-3 parity), 'half' = 1 pass; "
                   "mma_tflops = executed tensor-core rate of the WHOLE forward incl. all HBM-bound kernels and launch gaps")
    return res


def cudnn_same_gpu(B, dev, steps=8, warm=4):
    """The reference algorithm as plain PyTorch ops (cuDNN / cuBLAS / ATen library kernels) on THIS GPU -- what the reference's
    own nn.Modules dispatch to on the box (the reference package itself needs detectron2 / mmcv and cannot travel): the oracle
    restatement (pinned bit-exact to the live reference on CPU) on cuda, cudnn.benchmark = True
    (configs/_base_/common_base.py:16), fwd+bwd incl. losses, batch 64.  Variants: fp32 with TF32 convs (PyTorch default =
    the reference's out-of-the-box behaviour), + channels_last, + AMP fp16 autocast (the reference's SOLVER.AMP option)."""
    from gdr_net_b200 import synth
    from oracle import fixtures
    from oracle import gdrn_oracle as O

    torch.backends.cudnn.benchmark = True
    sd = synth.seeded_state_dict(fixtures.template_from_manifest(), 0)
    batch = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in synth.make_batch(B, seed=100, with_sym=WITH_SYM).items()}
    res = {}
    for name, cl, amp in (("tf32", False, False), ("tf32_channels_last", True, False), ("amp_fp16_channels_last", True, True)):
        leaf = {}
        for k, v in O.leaf_state_dict(sd, requires_grad=False).items():
            v = v.to(dev)
            if cl and v.dim() == 4:
                v = v.contiguous(memory_format=torch.channels_last)
            leaf[k] = v.requires_grad_(v.dtype.is_floating_point and "running" not in k)
        b = dict(batch)
        if cl:
            b["roi_img"] = b["roi_img"].contiguous(memory_format=torch.channels_last)

        def step():
            for v in leaf.values():
                if v.requires_grad:
                    v.grad = None
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                o = O.gdrn_forward(leaf, b, train=True, do_loss=True, pm_sym=bool(WITH_SYM))
            sum(o["losses"].values()).backward()

        for _ in range(warm):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        res[name] = {"value": round(B / ms * 1e3, 1), "unit": "crops/s", "ms_per_step": round(ms, 3)}
        del leaf
        torch.cuda.empty_cache()
    best = max(res.items(), key=lambda kv: kv[1]["value"])
    return {"variants": res, "best": best[0], "value": best[1]["value"], "unit": "crops/s",
            "what": "oracle restatement of the reference on cuda (cuDNN/cuBLAS/ATen), cudnn.benchmark=True, allow_tf32=" + str(torch.backends.cudnn.allow_tf32)
                    + f", fwd+bwd incl. losses and the reference's per-step host-side logging, batch {B}, {steps} timed steps",
            "cudnn": torch.backends.cudnn.version(), "torch": torch.__version__}


def cpu_baseline(sample_batch: int = 8, iters: int = 2, check=None):
    """The CPU oracle (port of the reference algorithm, pinned bit-exact to it: oracle/make_golden.py) timed on this
    box's host cores: train-mode fwd + bwd of a bounded sample of the same workload.  With `check` (the CUDA path's losses
    and logits of the B = 64 benchmark batch) the oracle is also run forward on that very batch and the outputs compared
    at north_star's 1e-3 (the checker role of the oracle; VERDICT r1 item 1)."""
    from gdr_net_b200 import synth
    from oracle import fixtures
    from oracle import gdrn_oracle as O

    cores = min(os.cpu_count() or 1, 32)  # more threads than this slow the oneDNN convolutions down on the 128-thread hosts
    torch.set_num_threads(cores)
    sd = synth.seeded_state_dict(fixtures.template_from_manifest(), 0)
    batch = synth.make_batch(sample_batch, seed=300)
    times = []
    for it in range(iters + 1):
        leaf = O.leaf_state_dict(sd)
        t0 = time.perf_counter()
        o = O.gdrn_forward(leaf, batch, train=True, do_loss=True)
        sum(o["losses"].values()).backward()
        dt = time.perf_counter() - t0
        if it > 0:
            times.append(dt)
    best = sum(times) / len(times)
    cb = {"value": round(sample_batch / best, 2), "unit": "crops/s", "cores": cores, "kind": "port",
          "sample": f"train-mode fwd+bwd of {sample_batch} crops x {iters} timed iterations (1 warm-up), torch CPU fp32, "
                    f"{cores} threads; per-crop rate of the batch-64 workload"}
    parity = None
    if check is not None:
        from gdr_net_b200.engine import LOSS_NAMES

        b64 = synth.make_batch(BATCH_PER_GPU, seed=100, with_sym=WITH_SYM)  # rank 0's benchmark batch
        t0 = time.perf_counter()
        with torch.no_grad():
            o = O.gdrn_forward(O.leaf_state_dict(sd, requires_grad=False), b64, train=True, do_loss=True, pm_sym=bool(WITH_SYM))
        t_fwd = time.perf_counter() - t0
        worst = 0.0
        for i, k in enumerate(LOSS_NAMES):
            ref = float(o["losses"][k])
            worst = max(worst, abs(float(check["losses"][i]) - ref) / abs(ref))
        head = check["logits"].view(BATCH_PER_GPU, 64, 64, 72)[..., :69].permute(0, 3, 1, 2).double()
        ref = o["head"].double()
        rel_l2 = float((head - ref).norm() / ref.norm())
        rel_max = float((head - ref).abs().max() / ref.abs().max())
        am, ram = head[:, 4:].argmax(1), ref[:, 4:].argmax(1)
        top2 = ref[:, 4:].topk(2, dim=1).values
        outside = int(((am != ram) & ((top2[:, 0] - top2[:, 1]) > 2e-3 * ref.abs().max())).sum())
        parity = {"mode": check["precision"], "batch": BATCH_PER_GPU, "tolerance": 1e-3,
                  "losses_max_rel": float(f"{worst:.3e}"), "head_rel_l2": float(f"{rel_l2:.3e}"), "head_rel_max": float(f"{rel_max:.3e}"),
                  "region_argmax_agreement": round(float((am == ram).double().mean()), 6),
                  "region_argmax_mismatches_outside_tie_margin": outside,
                  "oracle_fwd_s": round(t_fwd, 2),
                  "pass": bool(worst <= 1e-3 and rel_l2 <= 1e-3 and rel_max <= 2e-3 and outside == 0),
                  "what": "outputs of the last timed step of the headline mode (all 8 losses, the 69-channel head, region argmax) vs "
                          "the CPU oracle's train-mode forward on the same B=64 batch and weights"}
        if check["precision"] != "half":
            assert parity["pass"], f"B=64 parity check failed: {parity}"
    return cb, parity


def run_reference(args):
    """--impl reference: the reference's own algorithm on the host cores.  /root/reference does not travel to the GPU box,
    so this times the CPU oracle port (oracle/gdrn_oracle.py, pinned bit-exact against the live reference)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from gdr_net_b200 import synth
    from oracle import fixtures
    from oracle import gdrn_oracle as O

    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    sd = synth.seeded_state_dict(fixtures.template_from_manifest(), 0)
    sample = args.cpu_batch
    batch = synth.make_batch(sample, seed=300)

    def step():
        leaf = O.leaf_state_dict(sd)
        o = O.gdrn_forward(leaf, batch, train=True, do_loss=True)
        sum(o["losses"].values()).backward()

    steps, warm = args.steps, max(1, min(args.warmup, 2))
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    value = sample / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": "crops/s", "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": round(dt * 1e3, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1] (same as the CUDA arm); each step = a bounded sample of it", "parallelism": "host cpu"},
        "cpu_baseline": {"value": round(value, 2), "unit": "crops/s", "cores": cores, "kind": "port",
                         "sample": f"train-mode fwd+bwd of {sample} crops per step, torch CPU fp32, {cores} threads"},
        "e2e": {"value": round(value, 2), "unit": "crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--cpu-iters", type=int, default=1)
    ap.add_argument("--config", default="train", choices=["train", "ycbv", "pnp"],
                    help="train = BASELINE configs[1] (the headline; default), ycbv = configs[4] (B=32, symmetric PM), "
                         "pnp = configs[3] (stand-alone Patch-PnP, B=512)")
    ap.add_argument("--nin", type=int, default=69, choices=[67, 69], help="--config pnp: Patch-PnP input channels")
    ap.add_argument("--quick", action="store_true", help="device-timed value only (for profiler runs)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch every kernel from Python instead of one CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) to DIR/<name>.npy, float32/float64, at most 64 MB; "
                         "the train steps then use ordered (run-to-run reproducible) reductions instead of fp32 atomics")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA arm's outputs; the reference arm times a CPU sample of the workload")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
        if args.config == "pnp":
            run_pnp(args)
        else:
            run_ours(args)


if __name__ == "__main__":
    main()
