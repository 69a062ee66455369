"""Gradient with respect to the input clip, timed on the GPU (CUDA events): the stem's data gradient at 16 x 224^2 on the
tensor-core path (svit_patch_embed_s2d_dgrad + svit_d2s_clip) and on the col2im path (svit_gemm + svit_col2im3d, as the
fp32 parity mode runs it and with a bf16 gradient), and the clips/s of a frozen-model saliency pass (bf16 forward +
backward to the clip).  Prints one JSON object; --out also writes it to a file.

Rates: FLOP = 2 M 96 768 (M = cells = B Tc Hc Wc; N = 96 cell values, K = 8 taps x 96 channels, the MACs the dgrad
kernel issues); bytes = dY read (B L 96 bf16) + dclip written (B 3 T H W fp32).  The inputs are not flushed from L2
between iterations; at B = 8 the working set (dY, cells, dclip) is 154 MB, above the 126 MB of L2."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

KERNEL, STRIDE, PAD = (3, 7, 7), (2, 4, 4), (1, 3, 3)


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = None
    return info


def op_level(B, T, H, W, iters):
    from svit_b200 import ops

    g = torch.Generator().manual_seed(B)
    w = (torch.randn(96, 3, *KERNEL, generator=g) * 0.05).cuda()
    To, Ho, Wo = ((n + 2 * p - k) // s + 1 for n, k, s, p in zip((T, H, W), KERNEL, STRIDE, PAD))
    L = To * Ho * Wo
    Ntot = 1 + L + 4 * T
    dx16 = torch.randn(B, Ntot, 96, generator=g).to("cuda", torch.bfloat16)
    dx32 = dx16.float()
    shape = (B, 3, T, H, W)
    Tc, Hc, Wc = -(-T // STRIDE[0]), -(-H // STRIDE[1]), -(-W // STRIDE[2])
    M = B * Tc * Hc * Wc
    flop = 2.0 * M * 96 * 768
    nbytes = B * L * 96 * 2 + B * 3 * T * H * W * 4
    r = {"B": B, "clip": [T, H, W], "gflop": flop / 1e9, "mbytes_dy_read_plus_dclip_written": nbytes / 1e6}

    def rates(us):
        return {"us": round(us, 1), "tflops": round(flop / us / 1e6, 1), "gbps": round(nbytes / us / 1e3, 1)}

    tc = lambda: ops.input_grad_s2d(dx16, w, shape, torch.float32, KERNEL, STRIDE, PAD)
    r["tcgen05_dgrad_plus_d2s"] = rates(timed(tc, iters))
    # the two kernels on their own (the d2s on the cell gradient the dgrad left behind)
    ops.profile_start()
    for _ in range(iters):
        tc()
    prof = ops.profile_stop(iters)["detail"]
    for k, v in prof.items():
        if k.startswith("svit_patch_embed_s2d_dgrad"):
            r["dgrad_kernel"] = rates(v["ms_per_step"] * 1e3)
        elif k.startswith("svit_d2s_clip"):
            r["d2s_kernel_us"] = round(v["ms_per_step"] * 1e3, 1)
    ops.set_impl(gemm=ops.IMPL_SIMT)
    r["col2im_fp32_simt"] = rates(timed(lambda: ops.input_grad_col2im(dx32, w, shape, torch.float32, KERNEL, STRIDE, PAD),
                                        max(2, iters // 10), warmup=1))
    ops.set_impl(gemm=ops.IMPL_AUTO)
    r["col2im_bf16"] = rates(timed(lambda: ops.input_grad_col2im(dx16, w, shape, torch.float32, KERNEL, STRIDE, PAD),
                                   max(2, iters // 4), warmup=1))
    r["tcgen05_speedup_over_col2im_bf16"] = round(r["col2im_bf16"]["us"] / r["tcgen05_dgrad_plus_d2s"]["us"], 2)
    # agreement of the two paths on the same bf16 gradient (the col2im path accumulates in fp32 from the same bf16 inputs)
    a, b = tc(), ops.input_grad_col2im(dx16, w, shape, torch.float32, KERNEL, STRIDE, PAD)
    r["max_abs_diff_over_max_abs"] = ((a - b).abs().max() / b.abs().max()).item()
    return r


def saliency(B, iters):
    import svit_b200
    from svit_b200.config import ssv2_cfg

    torch.manual_seed(0)
    m = svit_b200.SViT(ssv2_cfg(), compute_dtype=torch.bfloat16).cuda().eval()
    m.requires_grad_(False)
    clip = torch.randn(B, 3, 16, 224, 224, device="cuda")

    def step():
        x = clip.clone().requires_grad_(True)
        probs = m([x])[0]
        probs.max(dim=1).values.sum().backward()
        return x.grad

    us = timed(step, iters, warmup=2)
    return {"B": B, "ms_per_pass": round(us / 1e3, 2), "clips_per_s": round(B / (us / 1e6), 1)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", type=int, nargs="+", default=[8, 64])
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--saliency-batch", type=int, default=8)
    ap.add_argument("--saliency-iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("input_grad_bench needs a CUDA device")
    res = {"gpu": gpu_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S"), "op": [], "saliency": None}
    for B in args.batches:
        res["op"].append(op_level(B, 16, 224, 224, args.iters))
        torch.cuda.empty_cache()
    res["saliency"] = saliency(args.saliency_batch, args.saliency_iters)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
