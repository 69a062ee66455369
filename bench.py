#!/usr/bin/env python
"""Benchmark of the SViT hot path on B200 (contract: see the task brief / DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, bf16, batch 64 clips / GPU)
  python bench.py --impl reference --gpus N --steps K ...  # reference arm: CPU oracle port on the host cores
  python bench.py ... --dump-outputs DIR                   # also write what the last timed forward computed, DIR/<name>.npy

One "step" = one forward of SViT (configs/ssv2.yaml geometry, random init) over one batch of synthetic
16x224^2 clips (BASELINE configs[1]).  `value` = clips/s with the batch resident in HBM; `e2e` = clips/s through the
public module call with pinned-host inputs (H2D of the clips and D2H of the class probabilities inside the timed region).
The same JSON line carries
  "train"              BASELINE configs[2]: the full training step (fwd + bwd + NCCL gradient all-reduce + clip + AdamW),
                       batch 8 clips / GPU, one CUDA graph per step -- the only leg with a collective, so this is the
                       number that shows multi-GPU communication cost in a --gpus N sweep;
  "torch_gpu_baseline" the reference's op sequence as stock PyTorch (autocast bf16) runs it on the same B200 (N = 1);
  "cpu_baseline"       the CPU oracle port on the host cores (N = 1).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ work model
def attn_flops(B, spec, thw, O_tot):
    """4*B*h*Nq*Nk*96 + 2*B*h*Lq*96*(kh+kw+kt)  (SURVEY.md 8d)."""
    T, H, W = thw
    sq, skv = spec["stride_q"][1], spec["stride_kv"][1]
    qh, qw = (H - 1) // sq + 1, (W - 1) // sq + 1
    kh, kw = (H - 1) // skv + 1, (W - 1) // skv + 1
    Lq, Lk = T * qh * qw, T * kh * kw
    Nq, Nk = 1 + Lq + O_tot, 1 + Lk + O_tot
    h = spec["num_heads"]
    return 4.0 * B * h * Nq * Nk * 96 + 2.0 * B * h * Lq * 96 * (kh + kw + T), [T, qh, qw], Nq, Nk


def work_per_clip(cfg):
    """Algorithmic FLOPs / bytes per clip for each kernel family (forward)."""
    from svit_b200.config import block_specs
    specs, patch_dims, _ = block_specs(cfg)
    O_tot = cfg.DATA.NUM_FRAMES * cfg.SVIT.O
    thw = list(patch_dims)
    L = thw[0] * thw[1] * thw[2]
    fl = {"attn": 0.0, "gemm": 2.0 * L * 96 * 441, "pool_bytes_bf16": 0.0}
    for sp in specs:
        N = 1 + thw[0] * thw[1] * thw[2] + O_tot
        C, D, h = sp["dim"], sp["dim_out"], sp["num_heads"]
        f, q_thw, Nq, Nk = attn_flops(1, sp, thw, O_tot)
        fl["attn"] += f
        fl["gemm"] += 2.0 * N * C * 3 * D + 2.0 * Nq * D * D + 2 * 2.0 * Nq * D * 4 * D
        if C != D:
            fl["gemm"] += 2.0 * N * C * D
        fl["pool_bytes_bf16"] += 2.0 * 96 * h * ((N + Nq) + 2 * (N + Nk))
        thw = q_thw
    return fl


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_forward_timing(max_seconds=25.0, max_runs=5):
    """Times the CPU oracle port of the reference forward (fp32, batch 1, all host threads).  Returns the run times, the
    thread count and the (probs, extra) of the last run."""
    from oracle import svit_oracle as O
    from svit_b200.config import block_specs, ssv2_cfg, state_shapes
    from tests.golden.recipe import synth_input, synth_state

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = ssv2_cfg()
    params = synth_state(state_shapes(cfg), 0, w_std=0.02)
    specs = block_specs(cfg)[0]
    clip = synth_input("bench.clip", (1, 3, 16, 224, 224), 1234)
    times = []
    t_begin = time.time()
    with torch.no_grad():
        out = O.svit_forward(clip, params, specs, cfg)  # warm-up
        while len(times) < max_runs and time.time() - t_begin < max_seconds:
            t0 = time.perf_counter()
            out = O.svit_forward(clip, params, specs, cfg)
            times.append(time.perf_counter() - t0)
    return times, cores, out


DUMP_LIMIT_BYTES = 64 << 20


def forward_outputs(probs, extra):
    """What a caller of the forward receives, under the names --dump-outputs writes."""
    d = {"forward_probs": probs}
    d.update({f"forward_{k}": v for k, v in extra.items() if torch.is_tensor(v)})
    return d


def dump_outputs(path, arrays):
    """Writes every array as <path>/<name>.npy in float32.  Above DUMP_LIMIT_BYTES in all, each array is replaced by the
    same fixed, seeded sample of its flattened elements, so two runs with the same arguments stay comparable element by
    element."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(4 * v.numel() for v in arrays.values())
    for name, v in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = v.numel() * DUMP_LIMIT_BYTES // total
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            v = v.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), v.numpy())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, cores, (probs, extra) = cpu_forward_timing(max_seconds=float("inf"), max_runs=args.steps + args.warmup)
    times = times[args.warmup:]
    sec = statistics.median(times)
    val = 1.0 / sec
    line = {"impl": "reference", "metric": "clips/sec (16x224^2, bf16) SViT forward", "value": val, "unit": "clips/s",
            "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "SViT ssv2.yaml forward, 16x224^2 clips, 4 object tokens/frame; each step = a "
                                   "batch-1 sample of the batch-64 workload on the host cores"},
            "cpu_baseline": {"value": val, "unit": "clips/s", "cores": cores, "kind": "port",
                             "sample": f"{len(times)} batch-1 forwards of the oracle port (torch CPU fp32)"},
            "e2e": {"value": val, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, forward_outputs(probs, extra))


# ------------------------------------------------------------------------------------------------ our arm
def _env():
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local_rank, dev


def _barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(ms, world, dev):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()
    return ms


def torch_gpu_forward_timing(dev, B=64, runs=5):
    """The honest same-box comparator (SURVEY 8d, BASELINE.md 3): the reference's forward as stock PyTorch runs it on
    this B200 -- ATen / cuBLAS / cuDNN kernels under torch.autocast(bf16), TF32 off, eager, batch B.  What is executed
    is the oracle port (oracle/svit_oracle.py: the reference's own op sequence, pinned to it by tests/golden); the
    unmodified reference modules are used instead when the tree is present (never on the GPU box).  Bench-only leg."""
    from oracle import svit_oracle as O
    from svit_b200.config import block_specs, ssv2_cfg, state_shapes
    from tests.golden.recipe import synth_state

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = ssv2_cfg()
    params = {k: v.to(dev) for k, v in synth_state(state_shapes(cfg), 0, w_std=0.02).items()}
    specs = block_specs(cfg)[0]
    gen = torch.Generator().manual_seed(4321)
    clip = torch.randn(B, 3, 16, 224, 224, generator=gen).to(dev)
    times = []
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for _ in range(2):
            O.svit_forward(clip, params, specs, cfg)
        torch.cuda.synchronize()
        for _ in range(runs):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            O.svit_forward(clip, params, specs, cfg)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
    del params, clip
    torch.cuda.empty_cache()
    return times


def train_leg(args, world, rank, dev, clocks_rank0=True):
    """configs[2]: the full training step -- forward + backward (bf16 activations, fp32 parameter gradients), the
    bucketed NCCL gradient all-reduce (world > 1), gradient clipping and the fused AdamW update -- batch 8 clips per GPU,
    replayed from ONE CUDA graph (svit_b200.GraphedTrainStep).  Returns the dict printed as "train" in the JSON line."""
    import svit_b200
    from svit_b200 import ops
    from svit_b200.config import ssv2_cfg
    from svit_b200.distributed import GradAllReducer
    from svit_b200.optim import construct_optimizer

    W, K = max(3, args.warmup), args.steps
    B = args.train_batch
    cfg = ssv2_cfg()
    torch.manual_seed(0)
    model = svit_b200.SViT(cfg, compute_dtype=torch.bfloat16).to(dev).train()
    reducer = GradAllReducer(model.parameters(), overlap=not args.no_overlap) if world > 1 else None
    optimizer = construct_optimizer(model, cfg)
    gen = torch.Generator().manual_seed(1234 + rank)
    clips = [torch.randn(B, 3, 16, 224, 224, generator=gen).to(torch.bfloat16).to(dev) for _ in range(2)]
    labels = torch.randint(0, cfg.MODEL.NUM_CLASSES, (B,), generator=gen).to(dev)
    launch = "cuda graph replay (forward + backward + all-reduce + clip + AdamW in one graph)"
    step = None
    if not args.no_graph:
        try:
            step = svit_b200.GraphedTrainStep(model, optimizer, clips[0], labels, reducer=reducer,
                                              max_norm=cfg.SOLVER.CLIP_GRAD_L2NORM, frames_pass=args.frames_pass)
        except Exception as e:  # the launch mechanism only: the same kernels run eagerly
            launch = f"eager (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
            step = None
            torch.cuda.synchronize()
    if step is None:
        if args.no_graph:
            launch = "eager"
        from svit_b200.distributed import consistency_loss, forward_video_frames

        def step(clip, lab):
            for p in model.parameters():
                p.grad = None
            if reducer is not None:
                reducer.prepare()
            preds, extra = model([clip])
            loss = torch.nn.functional.cross_entropy(extra["logits"].float(), lab)
            if args.frames_pass:
                _p, _e = forward_video_frames(model, clip)
                for k, v in consistency_loss(model._lambda, extra, _e).items():
                    loss = loss + model._lambda[k] * v
            loss.backward()
            if reducer is not None:
                reducer.finish()
            optimizer.step(max_norm=cfg.SOLVER.CLIP_GRAD_L2NORM)
            return loss.detach()

    for i in range(W):
        step(clips[i & 1], labels)
    _barrier(world)
    l0 = ops.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        loss = step(clips[i & 1], labels)
    e1.record()
    _barrier(world)
    ms = _max_over_ranks(e0.elapsed_time(e1), world, dev)
    launches = ops.launches() - l0
    loss_val = float(loss)
    out = {"metric": "clips/sec (16x224^2, bf16) SViT training step (fwd + bwd + grad all-reduce + clip + AdamW)",
           "value": world * B * K / (ms / 1e3), "unit": "clips/s", "ms_per_step": ms / K, "n_gpus": world,
           "batch_per_gpu": B, "global_batch": B * world, "steps": K, "warmup": W, "gpu_launches": launches,
           "launch": launch, "loss": loss_val,
           "allreduce_bytes_per_step": (reducer.bytes_per_step if reducer is not None else 0),
           "allreduce": ("none (1 GPU)" if reducer is None else
                         f"NCCL all-reduce (AVG) of {len(reducer.buckets)} fp32 buckets, "
                         + ("launched from backward as buckets complete" if reducer.overlap else "after backward")),
           "frames_pass": bool(args.frames_pass),
           "flops_per_clip": 3 * 138.16e9}
    out["tflops"] = out["value"] * out["flops_per_clip"] / 1e12 / world
    del step, model, optimizer, reducer, clips
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="svit_b200", choices=["svit_b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="clips per GPU (inference leg)")
    ap.add_argument("--train-batch", type=int, default=8, help="clips per GPU (training leg, configs[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step leg (configs[2])")
    ap.add_argument("--profile-json", default=None, help="write the per-kernel breakdown here")
    ap.add_argument("--lanes", type=int, default=int(os.environ.get("SVIT_FWD_LANES", "1")),
                    help="inference graph: independent sub-batches captured on separate streams")
    ap.add_argument("--no-graph", action="store_true", help="launch the kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-overlap", action="store_true", help="training leg: all-reduce after backward instead of overlapped")
    ap.add_argument("--host-input", default="uint8", choices=["uint8", "bf16"],
                    help="e2e leg: what crosses PCIe each step -- decoded uint8 frames [B,T,H,W,3] (normalised on the "
                         "device by svit_normalize_u8, datasets/utils.py:287-303) or pre-normalised bf16 clips")
    ap.add_argument("--frames-pass", action="store_true",
                    help="training leg: also run the reference's no-grad pass over the B*16 single frames "
                         "(TRAIN.FORWARD_VIDEO_FRAMES, tools/train_net.py:105-110)")
    ap.add_argument("--mode", default="both", choices=["both", "infer", "train"],
                    help="both: configs[1] headline + configs[2] as the 'train' object of the same JSON line; "
                         "train: only configs[2], printed as the main line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step of the timed forward legs (device-resident "
                         "and end-to-end) computed as DIR/<name>.npy (float32, at most 64 MB in all); the inputs are "
                         "seeded, so runs with the same arguments write the same arrays")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # The training step is not a reproducible function of its inputs: its backward sums gradients with fp32 atomics in
    # no fixed order, and the bf16 weight copies carry those last-bit differences into every later step.
    if args.dump_outputs and args.mode == "train" and args.impl != "reference":
        ap.error("--dump-outputs writes the forward legs' outputs; --mode train runs none")
    if args.impl == "reference":
        return run_reference(args)
    if args.mode == "train":
        return run_train(args)

    import torch.distributed as dist

    import svit_b200
    from svit_b200 import ops
    from svit_b200.config import ssv2_cfg

    world, rank, local_rank, dev = _env()
    W = max(3, args.warmup)
    K = args.steps
    B = args.batch
    cfg = ssv2_cfg()
    torch.manual_seed(0)
    model = svit_b200.SViT(cfg, compute_dtype=torch.bfloat16).to(dev).eval()
    gen = torch.Generator().manual_seed(1234 + rank)
    host = [torch.randn(B, 3, 16, 224, 224, generator=gen).to(torch.bfloat16).pin_memory() for _ in range(2)]
    dev_in = [h.to(dev, non_blocking=True) for h in host]
    probs_host = torch.empty(B, cfg.MODEL.NUM_CLASSES, dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    # The forward is captured once in a CUDA graph (svit_b200.GraphedForward) and replayed: one graph launch per step
    eager = model
    model_u8 = None
    if not args.no_graph:
        model = svit_b200.GraphedForward(eager, dev_in[0], lanes=args.lanes)
        if args.host_input == "uint8":
            # the end-to-end leg's graph takes the decoded frames themselves: the colour normalisation is fused into the
            # cell-layout kernel of the patch embed (svit_s2d_clip, in_kind uint8), no bf16 clip is ever materialised.
            # Captured here, next to the first graph and before any collective of the timed legs.
            model_u8 = svit_b200.GraphedForward(
                eager, torch.zeros(B, 16, 224, 224, 3, dtype=torch.uint8, device=dev), lanes=args.lanes)
    # ---- device-resident throughput
    with torch.no_grad():
        for i in range(W):
            model([dev_in[i & 1]] if args.no_graph else dev_in[i & 1])
        _barrier(world)
        if rank == 0:
            sampler.start()
        l0 = ops.launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            out, extra = model([dev_in[i & 1]] if args.no_graph else dev_in[i & 1])
        e1.record()
        _barrier(world)
        ms = _max_over_ranks(e0.elapsed_time(e1), world, dev)
        launches = ops.launches() - l0
        # copied now: the graph's static outputs are overwritten by the next replay
        outputs = ({k: v.cpu() for k, v in forward_outputs(out, extra).items()}
                   if args.dump_outputs and rank == 0 else None)

        # ---- end to end: pinned host clips -> H2D (copy stream, double buffered) -> forward -> D2H of the probabilities
        copy_stream = torch.cuda.Stream(device=dev)
        main_stream = torch.cuda.current_stream()
        u8 = args.host_input == "uint8"
        if u8:  # frames as the decoder leaves them (datasets/utils.py:287-303 runs on the device, inside the stem)
            host = [torch.randint(0, 256, (B, 16, 224, 224, 3), generator=gen, dtype=torch.uint8).pin_memory()
                    for _ in range(2)]
        staged = [torch.empty(host[0].shape, dtype=host[0].dtype, device=dev) for _ in range(2)]
        mean, std = cfg.DATA.MEAN, cfg.DATA.STD

        def model_e2e(inp):
            if args.no_graph:
                return model([inp[0]])  # SViT.forward accepts uint8 [B, T, H, W, 3]
            return model_u8(inp) if u8 else model(inp)
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]

        def e2e_loop(n):
            for i in range(n):
                j = i & 1
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(freed[j])
                    staged[j].copy_(host[j], non_blocking=True)
                    ready[j].record(copy_stream)
                main_stream.wait_event(ready[j])
                out, _ = model_e2e([staged[j]] if args.no_graph else staged[j])
                freed[j].record(main_stream)
                probs_host.copy_(out, non_blocking=True)

        for j in range(2):
            freed[j].record(main_stream)
        e2e_loop(2)
        _barrier(world)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        copy_stream.wait_event(s0)
        e2e_loop(K)
        main_stream.wait_stream(copy_stream)
        s1.record()
        _barrier(world)
        ms_e2e = _max_over_ranks(s0.elapsed_time(s1), world, dev)
        clocks = sampler.stop() if rank == 0 else None
        if outputs is not None:
            outputs["e2e_probs"] = probs_host.clone()

        # ---- per-kernel breakdown (separate instrumented pass, CUDA events around every C-ABI call)
        prof = None
        if rank == 0:
            ops.profile_start()
            for i in range(2):
                eager([dev_in[i & 1]])
            torch.cuda.synchronize()
            prof = ops.profile_stop(steps=2)

    value = world * B * K / (ms / 1e3)
    e2e_val = world * B * K / (ms_e2e / 1e3)
    h2d_bytes = host[0].numel() * host[0].element_size()

    # ---- training-step leg (configs[2]): every rank takes part (this is the leg with the collective)
    del model, eager, staged, dev_in, host
    torch.cuda.empty_cache()
    _barrier(world)
    train = None
    if not args.no_train:
        tsampler = ClockSampler(local_rank)
        if rank == 0:
            tsampler.start()
        train = train_leg(args, world, rank, dev)
        if rank == 0:
            train["clocks"] = tsampler.stop()

    if rank != 0:
        if world > 1:
            dist.barrier()  # stay alive until rank 0 has finished its single-rank legs: ordered NCCL teardown
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    wk = work_per_clip(cfg)
    fam = prof["families"]
    tot_ms = sum(f["ms_per_step"] for f in fam.values())
    # denominators: the BURST bf16 figure (SURVEY 8d default); the sustained one is reported beside it
    tf_burst = peaks["bf16_tflops"]
    tf_sust = peaks.get("bf16_tflops_sustained", tf_burst)

    def tensor_roof(name, flops_per_clip):
        t = fam.get(name, {}).get("ms_per_step", 0.0)
        ach = flops_per_clip * B / (t / 1e3) / 1e12 if t > 0 else 0.0
        return {"bound": "tensor", "achieved": ach, "peak": tf_burst, "unit": "TFLOP/s", "frac": ach / tf_burst,
                "frac_of_sustained": ach / tf_sust, "peak_sustained": tf_sust,
                "traffic": None, "kernel": name, "share_of_step": t / tot_ms if tot_ms else None,
                "peak_source": f"{peaks['_source']} (burst bf16 GEMM)"}

    roof_attn = tensor_roof("attention", wk["attn"])
    roof_gemm = tensor_roof("gemm", wk["gemm"])
    t_pool = fam.get("pool_ln", {}).get("ms_per_step", 0.0)
    ach_pool = wk["pool_bytes_bf16"] * B / (t_pool / 1e3) / 1e9 if t_pool > 0 else 0.0
    roof_pool = {"bound": "hbm", "achieved": ach_pool, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                 "frac": ach_pool / peaks["hbm_gbs"], "traffic": None, "kernel": "pool_ln",
                 "share_of_step": t_pool / tot_ms if tot_ms else None, "peak_source": peaks["_source"]}
    traffic_path = os.path.join(ROOT, "profiles", "traffic.json")
    tr = json.load(open(traffic_path)) if os.path.exists(traffic_path) else {}
    for r in (roof_attn, roof_gemm, roof_pool):
        r["traffic"] = tr.get(r["kernel"])
    # dominant KERNEL = the C-ABI call (one kernel shape) with the largest share of the step -- GEMM, attention or
    # pooling; its roofline is algorithmic work per launch / average launch duration (CUDA events, instrumented pass)
    import re
    best = None
    O_tot = cfg.DATA.NUM_FRAMES * cfg.SVIT.O
    for tag, d in prof["detail"].items():
        per_launch_ms = d["ms_per_step"] / max(d["calls_per_step"], 1e-9)
        m = re.match(r"svit_gemm\[(\d+)x(\d+)x(\d+)\]", tag)
        a = re.match(r"svit_attn_fwd\[B(\d+) h(\d+) Nq(\d+) Nk(\d+)\]", tag)
        pl = re.match(r"svit_pool_ln_fwd\[\w B(\d+) h(\d+) (\d+)x(\d+)x(\d+) s(\d+)\]", tag)
        mf = re.match(r"svit_mlp_fused\[(\d+)x(\d+)x(\d+)x(\d+)\]", tag)
        if m:
            M_, N_, K_ = (int(x) for x in m.groups())
            work, bound = 2.0 * M_ * N_ * K_, "tensor"
        elif mf:  # fc1 + fc2 in one kernel: [M x C x H x N]
            M_, C_, H_, N_ = (int(x) for x in mf.groups())
            work, bound = 2.0 * M_ * H_ * (C_ + N_), "tensor"
        elif a:
            B_, h_, Nq_, Nk_ = (int(x) for x in a.groups())
            work, bound = 4.0 * B_ * h_ * Nq_ * Nk_ * 96, "tensor"
        elif pl:
            B_, h_, T_, H_, W_, s_ = (int(x) for x in pl.groups())
            n_in = 1 + T_ * H_ * W_ + O_tot
            n_out = 1 + T_ * ((H_ - 1) // s_ + 1) * ((W_ - 1) // s_ + 1) + O_tot
            work, bound = 2.0 * 96 * B_ * h_ * (n_in + n_out), "hbm"
        else:
            continue
        if best is None or d["ms_per_step"] > best[1]["ms_per_step"]:
            best = (tag, d, work, bound, per_launch_ms)
    dominant = max((roof_attn, roof_gemm, roof_pool), key=lambda r: r["share_of_step"] or 0.0)
    if best is not None:
        tag, d, work, bound, per_launch_ms = best
        if bound == "tensor":
            ach = work / (per_launch_ms / 1e3) / 1e12
            dominant = {"bound": bound, "achieved": ach, "peak": tf_burst, "unit": "TFLOP/s", "frac": ach / tf_burst,
                        "frac_of_sustained": ach / tf_sust, "peak_sustained": tf_sust,
                        "peak_source": f"{peaks['_source']} (burst bf16 GEMM; sustained beside it)"}
        else:
            ach = work / (per_launch_ms / 1e3) / 1e9
            dominant = {"bound": bound, "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": ach / peaks["hbm_gbs"], "peak_source": peaks["_source"]}
        dominant.update({"traffic": tr.get(tag), "kernel": tag, "launches_per_step": d["calls_per_step"],
                         "avg_launch_ms": per_launch_ms, "work_per_launch": work,
                         "share_of_step": d["ms_per_step"] / tot_ms if tot_ms else None})

    line = {"metric": "clips/sec (16x224^2, bf16) SViT forward", "value": value, "unit": "clips/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"SViT (configs/ssv2.yaml: MViTv2-S 16x224^2 + 4 object tokens/frame) inference forward, "
                                   f"batch {B} clips per GPU, random init",
                       "parallelism": f"dp{world}", "global_batch": B * world,
                       "l2_policy": "inputs larger than L2 (308 MB of bf16 clips per step, >1 GB activations)",
                       "host_input_dtype": args.host_input, "launch": "eager" if args.no_graph else "cuda graph replay",
                       "train_leg": "configs[2] (training step with the gradient all-reduce) is the 'train' object of "
                                    "this line: the only leg with a collective"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e_val, "unit": "clips/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": probs_host.numel() * probs_host.element_size()},
            "roofline": dominant, "roofline_attention": roof_attn, "roofline_gemm": roof_gemm,
            "roofline_pool_ln": roof_pool,
            "kernel_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in sorted(fam.items())}}
    if train is not None:
        line["train"] = train
    if world == 1 and not args.no_torch_gpu_baseline:
        try:
            tt = torch_gpu_forward_timing(dev, B=B)
            med = statistics.median(tt)
            line["torch_gpu_baseline"] = {
                "value": B / (med / 1e3), "unit": "clips/s", "ms_per_step": med, "batch": B,
                "what": "reference op sequence (oracle port) as stock PyTorch eager on this B200: torch.autocast(bf16), "
                        "TF32 off, ATen / cuBLAS / cuDNN kernels, inputs resident in HBM",
                "speedup_vs_torch_gpu": value / (B / (med / 1e3))}
        except Exception as e:
            line["torch_gpu_baseline"] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    if world == 1 and not args.no_cpu_baseline:
        times, cores, _ = cpu_forward_timing(max_seconds=20.0, max_runs=5)
        sec = statistics.median(times)
        line["cpu_baseline"] = {"value": 1.0 / sec, "unit": "clips/s", "cores": cores, "kind": "port",
                                "sample": f"{len(times)} batch-1 fp32 forwards of the CPU oracle port "
                                          f"(1 of the {B} clips of a step), median {sec:.3f} s"}
    if args.profile_json:
        with open(args.profile_json, "w") as f:
            json.dump(prof, f, indent=1)
    print(json.dumps(line), flush=True)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_train(args):
    """--mode train: configs[2] alone, printed as the main JSON line."""
    import torch.distributed as dist

    world, rank, local_rank, dev = _env()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t = train_leg(args, world, rank, dev)
    if rank == 0:
        line = {"metric": t["metric"], "value": t["value"], "unit": "clips/s", "n_gpus": world, "steps": t["steps"],
                "warmup": t["warmup"], "ms_per_step": t["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "gpu_launches": t["gpu_launches"],
                "loss": t["loss"], "clocks": sampler.stop(),
                "config": {"workload": f"SViT (configs/ssv2.yaml) training step, batch {t['batch_per_gpu']} clips per GPU, "
                                       "random init, cross-entropy on the class logits, fused clip_grad_norm + AdamW step"
                                       + (", + no-grad frames pass (B*16 frames, T=1)" if args.frames_pass else ""),
                           "parallelism": f"dp{world}", "global_batch": t["global_batch"], "launch": t["launch"],
                           "allreduce": t["allreduce"], "allreduce_bytes_per_step": t["allreduce_bytes_per_step"]}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
