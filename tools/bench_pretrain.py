"""Stage-1 (TSFormer pre-training) step benchmark: TSFormer.pretrain_precision "fp32" vs "bf16" in one process.

One training step = pretrain forward (dropout live) + masked MAE + backward + FusedClipAdam.step, on a fixed device-resident
batch with the synthetic TSFormer weights.  Both modes are timed alternately, step by step, with CUDA events after warm-up
of each mode.  Prints one JSON line per workload with samples/s, ms/step and the implied seconds per pre-training epoch.

--profile DIR: a separate torch.profiler run (profiler on, so not a timing run) that writes per-kernel CUDA time per step of
both modes to DIR/pretrain_kernels.txt and reports the attention kernels' useful TFLOP/s computed from the shapes.

Usage:  python tools/bench_pretrain.py [--steps 20] [--warmup 3] [--workloads METR-LA,PEMS04] [--profile DIR]
"""
import argparse
import json
import os
import random
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# name -> (batch size, nodes, patches, public series length in steps); the shipped TSFormer_<NAME>.py batch sizes are
# not used: B is the issue-sized step (B = 8 / 6) so that both modes fit comfortably next to each other
WORKLOADS = {"METR-LA": (8, 207, 168, 34272), "PEMS04": (6, 307, 336, 16992)}
ATTN_KERNELS = {"fp32": ("attn_fwd_kernel", "attn_bwd_q_kernel", "attn_bwd_kv_kernel"),
                "bf16": ("tc_attn_train_fwd_kernel", "tc_attn_train_bwd_kernel", "tc_attn_pack_kernel")}


def train_windows(series_len, P):
    """Pre-training windows per epoch: a 70 % train split of the series, one window per start with a full history of P
    patches and 12 future steps (derived from the public series length; the raw data is not in the repository)."""
    return int(0.7 * (series_len - P * 12 - 12 + 1))


def attention_flops(S, nu, P):
    """Useful attention FLOPs of one step from the shapes: 4 encoder layers over nu tokens + 1 decoder layer over P tokens,
    4 heads of 24: forward 2 GEMMs (QK^T, PV), backward 5 (S recomputed, dP, dV, dK, dQ); 2 FLOPs per multiply-add."""
    per = lambda n: 2.0 * S * 4 * n * n * 24          # noqa: E731  one [n x n x 24] GEMM per (sequence, head)
    fwd = 2 * (4 * per(nu) + per(P))
    bwd = 5 * (4 * per(nu) + per(P))
    return fwd, bwd


def build(name, device):
    from oracle import step_oracle as O
    from step.step_arch import TSFormer
    from step_b200.optim import FusedClipAdam
    B, N, P, _ = WORKLOADS[name]
    model = TSFormer(patch_size=12, in_channel=1, embed_dim=96, num_heads=4, mlp_ratio=4, dropout=0.1, num_token=float(P),
                     mask_ratio=0.75, encoder_depth=4, decoder_depth=1, mode="pre-train")
    model.load_state_dict(O.synthetic_tsformer_params(0), strict=True)
    model = model.to(device).train()
    random.seed(0)
    model.mask()
    model.mask.fixed = (model.mask.unmasked_tokens, model.mask.masked_tokens)
    history = torch.randn(B, P * 12, N, 1, generator=torch.Generator().manual_seed(1)).to(device)
    opt = FusedClipAdam([p for p in model.parameters() if p.requires_grad], lr=5e-4, weight_decay=1e-5, max_norm=5.0)
    return model, history, opt


def step(model, history, opt, precision):
    from step.step_loss.step_loss import masked_mae
    model.pretrain_precision = precision
    model.zero_grad(set_to_none=True)
    rec, label = model(history_data=history)
    loss = masked_mae(rec, label, null_val=0.0)
    loss.backward()
    opt.step()
    return loss


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power, clock = [x.strip() for x in out[0].split(",")]
    except Exception as e:                     # noqa: BLE001 - report, do not guess
        power, clock = f"unavailable ({type(e).__name__})", "unavailable"
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_modes(name, steps, warmup, device):
    model, history, opt = build(name, device)
    B, N, P, series = WORKLOADS[name]
    for prec in ("fp32", "bf16"):
        for _ in range(warmup):
            step(model, history, opt, prec)
    torch.cuda.synchronize()
    ms = {"fp32": [], "bf16": []}
    losses = {"fp32": [], "bf16": []}
    for _ in range(steps):
        for prec in ("fp32", "bf16"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            loss = step(model, history, opt, prec)
            e1.record()
            torch.cuda.synchronize()
            ms[prec].append(e0.elapsed_time(e1))
            losses[prec].append(loss.item())
    windows = train_windows(series, P)
    res = {"workload": f"TSFormer_{name}", "B": B, "N": N, "P": P, "steps": steps, "warmup": warmup,
           "train_windows_per_epoch": windows}
    for prec in ("fp32", "bf16"):
        t = sorted(ms[prec])
        med = t[len(t) // 2]
        sps = B / (med / 1e3)
        res[prec] = {"ms_per_step_median": round(med, 3), "ms_per_step_min": round(t[0], 3), "ms_per_step_max": round(t[-1], 3),
                     "samples_per_s": round(sps, 1), "s_per_epoch": round(windows / sps, 1),
                     "loss_finite": all(x == x and abs(x) < float("inf") for x in losses[prec])}
    res["speedup_bf16_over_fp32"] = round(res["fp32"]["ms_per_step_median"] / res["bf16"]["ms_per_step_median"], 3)
    return res


def profile_modes(name, device, out_dir, steps=3):
    from torch.profiler import ProfilerActivity, profile
    model, history, opt = build(name, device)
    B, N, P, _ = WORKLOADS[name]
    lines, summary = [], {}
    for prec in ("fp32", "bf16"):
        for _ in range(2):
            step(model, history, opt, prec)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                step(model, history, opt, prec)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if t > 0:
                per[ev.key] = per.get(ev.key, 0.0) + t / 1e3 / steps            # ms per step
        total = sum(per.values())
        attn = sum(v for k, v in per.items() if any(a in k for a in ATTN_KERNELS[prec]))
        fwd_f, bwd_f = attention_flops(B * N, len(model.mask.unmasked_tokens), P)
        summary[prec] = {"gpu_ms_per_step": round(total, 3), "attention_ms_per_step": round(attn, 3),
                         "attention_share": round(attn / total, 3),
                         "attention_useful_tflops": round((fwd_f + bwd_f) / (attn / 1e3) / 1e12, 2)}
        lines.append(f"== TSFormer_{name} B={B} N={N} P={P}  pretrain_precision={prec}: {total:.3f} ms of kernels per step, "
                     f"attention {attn:.3f} ms ({100 * attn / total:.1f} %), useful attention FLOPs "
                     f"{(fwd_f + bwd_f) / 1e9:.1f} G/step -> {summary[prec]['attention_useful_tflops']} TFLOP/s")
        for k, v in sorted(per.items(), key=lambda kv: -kv[1])[:25]:
            lines.append(f"  {v:9.3f} ms  {100 * v / total:5.1f} %  {k[:150]}")
    with open(os.path.join(out_dir, f"pretrain_kernels_{name}.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    return summary


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default="METR-LA,PEMS04")
    ap.add_argument("--profile", default=None, help="directory for the torch.profiler per-kernel summary")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if not torch.cuda.is_available():
        sys.exit("bench_pretrain.py measures the GPU: no CUDA device found")
    from step_b200 import build as step_build
    step_build.build()
    device = torch.device("cuda", 0)
    info = gpu_info()
    for name in args.workloads.split(","):
        res = time_modes(name, args.steps, args.warmup, device)
        res.update(info)
        if args.profile:
            os.makedirs(args.profile, exist_ok=True)
            res["profile"] = profile_modes(name, device, args.profile)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
