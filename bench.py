#!/usr/bin/env python
"""STEP fwd+bwd throughput benchmark (BASELINE.json metric) - see the contract in DESIGN.md section 6.

  python bench.py --gpus 1 --steps 10 --warmup 3            # our B200-native path
  python bench.py --impl reference --steps 2 --warmup 1     # the reference algorithm on the host CPU cores
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W               # one rank per GPU, batch-parallel
  ... bench.py --gpus N --workload PEMS07 --mode node         # node-sharded TSFormer + one NCCL all-gather
  python bench.py --steps 10 --warmup 3 --dump-outputs DIR  # + the last timed step's outputs and gradients as .npy

A "step" = one training step of STEP_<workload> (METR-LA: N=207 nodes, per-GPU batch 32, 168 patches of 12 = 2016-step
long history): forward (frozen TSFormer in train() exactly as the reference runs it, discrete graph learning, Graph
WaveNet), step_loss, backward to every trainable parameter (+ NCCL gradient all-reduce when N > 1).  Synthetic N(0,1)
inputs, real pre-trained TSFormer weights for METR-LA (tests/golden fixture), seeded random GWNet/DGL weights; dropout
and Gumbel seeds derive from a fixed torch seed, so the same arguments give the same inputs in every run.
Prints ONE JSON line.
"""
import argparse
import json
import os
import pickle
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# (nodes, per-GPU batch, patches) of the reference's STEP_<NAME>.py configs (SURVEY section 8)
WORKLOADS = {"METR-LA": (207, 32, 168), "PEMS04": (307, 8, 336), "PEMS-BAY": (325, 32, 168), "PEMS07": (883, 4, 168)}
# --dump-outputs: the largest array (discrete_graph_learning.fc.weight's gradient, 38 M values at METR-LA) is sampled
DUMP_MAX_ELEMS = 1 << 21
DUMP_MAX_BYTES = 64 << 20


def metric_name(ds):
    n, b, _ = WORKLOADS[ds]
    return "STEP fwd+bwd samples/sec (STEP_%s, N=%d, per-GPU batch %d, 12->12)" % (ds, n, b)


def ts_args(patches):
    return dict(patch_size=12, in_channel=1, embed_dim=96, num_heads=4, mlp_ratio=4, dropout=0.1, num_token=float(patches),
                mask_ratio=0.75, encoder_depth=4, decoder_depth=1, mode="forecasting")


def gw_args(nodes):
    return dict(num_nodes=nodes, support_len=2, dropout=0.3, gcn_bool=True, addaptadj=True, aptinit=None, in_dim=2, out_dim=12,
                residual_channels=32, dilation_channels=32, skip_channels=256, end_channels=512, kernel_size=2, blocks=4, layers=2)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the config's, 32 for METR-LA)")
    ap.add_argument("--workload", default="METR-LA", choices=sorted(WORKLOADS),
                    help="STEP config to run; METR-LA is the headline (BASELINE.json configs[1])")
    ap.add_argument("--mode", default="batch", choices=["batch", "node"],
                    help="multi-GPU partitioning: batch-parallel (each rank its own batch, NCCL gradient all-reduce) or "
                         "node-parallel (every rank encodes its node range of the SAME batch, one NCCL all-gather of the "
                         "TSFormer states before the N x N similarity; BASELINE.json configs[4])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the PyTorch-eager-on-this-GPU comparator")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--only-resident", action="store_true", help="profiling aid: run only the device-resident loop")
    ap.add_argument("--no-dropout", action="store_true", help="parity-style run (all dropout off); not the headline")
    ap.add_argument("--precision", default=os.environ.get("STEP_B200_PRECISION", "bf16"), choices=["bf16", "fp32"],
                    help="TSFormer encoder kernels: bf16 tcgen05 tensor cores (default, BASELINE config) or fp32 CUDA cores")
    ap.add_argument("--chunk-seqs", type=int, default=int(os.environ.get("STEP_B200_TS_CHUNK", "0")))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (y_hat, theta, adj_knn, gsl_coefficient, "
                         "loss and every trainable parameter's gradient) as DIR/<name>.npy in float32, so that two builds "
                         "can be compared output for output; arrays over %d elements are written as a fixed sample"
                         % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# --------------------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        time.sleep(0.05)
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def profile_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum of the first kernel in a committed `tools/ncu_summary.py` text
    (profiles/<name>), in bytes; None if the file is absent."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None
    tot, seen = 0.0, set()
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for line in open(path):
        m = re.match(r"\s*(dram__bytes_(read|write)\.sum)\s+([\d.,]+)\s+(\w+)", line)
        if m and m.group(1) not in seen:
            seen.add(m.group(1))
            tot += float(m.group(3).replace(",", "")) * unit.get(m.group(4), 1.0)
    return tot if len(seen) == 2 else None


def write_dataset(tmp, ds, node_feats):
    d = os.path.join(tmp, "datasets", ds)
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "data_in12_out12.pkl"), "wb") as f:
        pickle.dump({"processed_data": node_feats.unsqueeze(-1).numpy()}, f)


def ts_state(ds):
    if ds != "METR-LA":        # only the METR-LA checkpoint is small enough to ship as a fixture
        from step_b200 import synth
        return synth.synthetic_tsformer_params(1)
    return torch.load(os.path.join(ROOT, "tests", "golden", "tsformer_METR-LA_state.pt"))


def dump_sample(t):
    """t itself, or, above DUMP_MAX_ELEMS elements, one element of every stride-wide window of the flattened tensor at
    offsets drawn from a generator seeded by its size: every run and every build samples the same entries."""
    t = t.detach()
    n = t.numel()
    if n <= DUMP_MAX_ELEMS:
        return t
    stride = n // DUMP_MAX_ELEMS
    g = torch.Generator().manual_seed(n)
    idx = torch.arange(DUMP_MAX_ELEMS) * stride + torch.randint(stride, (DUMP_MAX_ELEMS,), generator=g)
    return t.reshape(-1)[idx.to(t.device)]


def dump_outputs(arm, out_dir):
    """Writes what the arm's last train_step handed its caller: the model's 4-tuple, the loss and the gradient of every
    trainable parameter (the fp32 values an optimiser step would consume)."""
    y_hat, theta, adj_knn, coeff, loss = arm.last_outputs
    arrays = {"y_hat": y_hat, "theta": theta, "adj_knn": adj_knn, "gsl_coefficient": torch.tensor(coeff), "loss": loss}
    for name, p in arm.model.named_parameters():
        if p.grad is not None:
            arrays["grad." + name] = p.grad
    arrays = {k: dump_sample(v).to(torch.float32).cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    sys.stderr.write("bench.py: %d arrays, %.1f MB written to %s\n" % (len(arrays), total / 1e6, out_dir))


# --------------------------------------------------------------------------------------------- CPU comparator
def cpu_reference_run(ds, steps, warmup, batch, dropout=True):
    """The reference's CPU path on the host cores, run through oracle/step_oracle.py's restatement of its torch modules
    (kind "port"; tests/test_oracle_golden.py holds the restatement to the reference's own outputs).  Same config except
    a bounded per-step batch.  Returns (samples/s, info)."""
    from oracle import step_oracle as O
    nodes, _, patches = WORKLOADS[ds]
    # torch CPU ops on these shapes slow down badly past ~16-32 threads (measured on the 128-thread GPU host:
    # 83 s/step with 128 threads); use the best-performing setting and report it as `cores`
    torch.set_num_threads(min(os.cpu_count() or 1, int(os.environ.get("STEP_B200_CPU_THREADS", "32"))))
    params = O.synthetic_trainable_params(ds, 0)
    sd = dict(params)
    sd.update(O.bn_buffers(ds))
    sd.update({"tsformer." + k: v for k, v in ts_state(ds).items()})
    node_feats = O.synthetic_node_feats(ds, 0)
    history, long_history, future, uniform = O.synthetic_batch(ds, batch, patches, 0)
    times = []
    for k in params:
        sd[k] = sd[k].clone().requires_grad_(True)
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss, _ = O.train_step(sd, history, long_history, future, node_feats, uniform, epoch=1, null_val=0.0,
                               gw_drop=0.3 if dropout else 0.0, ts_drop=0.1 if dropout else 0.0)
        loss.backward()
        for k in params:
            sd[k].grad = None
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    what = "oracle/step_oracle.py (restatement of the reference's torch modules)"
    return batch / dt, {"cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"{steps} timed fwd+bwd steps (after {warmup} warm-up) of STEP_{ds} at batch {batch} "
                                  f"(CPU samples/s is ~flat in batch), fp32, dropout {'live as in the reference train()' if dropout else 'off'}, "
                                  f"{dt:.2f} s/step; {what}"}


def gpu_eager_baseline(ds, batch, dev, steps=3, warmup=2):
    """SURVEY section 8(d)(iv): the reference's modules under PyTorch eager on THIS GPU - the same-box comparator the
    reference would run on a B200.  Executed through oracle/step_oracle.py's functional restatement of those modules
    (cuBLAS / ATen kernels, F.scaled_dot_product_attention as nn.TransformerEncoderLayer dispatches it), fp32 with
    TF32 off and bf16 autocast, dropout live, same batch.  The oracle is only the comparator here."""
    from oracle import step_oracle as O
    nodes, _, patches = WORKLOADS[ds]
    params = O.synthetic_trainable_params(ds, 0)
    sd = dict(params)
    sd.update(O.bn_buffers(ds))
    sd.update({"tsformer." + k: v for k, v in ts_state(ds).items()})
    sd = {k: v.to(dev) for k, v in sd.items()}
    for k in params:
        sd[k].requires_grad_(True)
    node_feats = O.synthetic_node_feats(ds, 0).to(dev)
    history, long_history, future, uniform = (t.to(dev) for t in O.synthetic_batch(ds, batch, patches, 0))
    out = {}
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, O.USE_SDPA)
    O.USE_SDPA = True
    try:
        for name in ("fp32", "bf16_autocast"):
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            try:
                def step():
                    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(name == "bf16_autocast")):
                        loss, _ = O.train_step(sd, history, long_history, future, node_feats, uniform, epoch=1, null_val=0.0,
                                               gw_drop=0.3, ts_drop=0.1)
                    loss.backward()
                    for k in params:
                        sd[k].grad = None
                for _ in range(warmup):
                    step()
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    step()
                e1.record()
                torch.cuda.synchronize(dev)
                ms = e0.elapsed_time(e1) / steps
                out[name] = {"value": batch / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms}
            except Exception as e:      # noqa: BLE001  (e.g. out of memory at a large config: report, do not die)
                out[name] = {"error": repr(e)[:200]}
                torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, O.USE_SDPA = prev
    out["what"] = ("oracle/step_oracle.py restatement of the reference's torch modules run by PyTorch %s eager on this GPU "
                   "(F.linear / SDPA / conv1d / einsum library kernels), STEP_%s batch %d, dropout live, %d timed steps"
                   % (torch.__version__, ds, batch, steps))
    del sd
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------- our arm
class Arm:
    """One configured workload on this rank: model, reducer, host / resident batches and the step function."""

    def __init__(self, ds, batch, mode, precision, dev, rank, world, no_dropout=False, chunk_seqs=0):
        from step_b200 import parallel, synth as O      # deterministic synthetic tensors (never the oracle)
        from step.step_arch import STEP
        from step.step_loss import step_loss
        self.ds, self.B, self.mode, self.dev, self.rank, self.world = ds, batch, mode, dev, rank, world
        self.nodes, _, self.patches = WORKLOADS[ds]
        self.step_loss = step_loss
        self.overlap = False
        node_feats = O.synthetic_node_feats(ds, 0)
        tmp = tempfile.mkdtemp(prefix="step_bench_")
        write_dataset(tmp, ds, node_feats)
        torch.save({"model_state_dict": ts_state(ds)}, os.path.join(tmp, "ts.pt"))
        cwd = os.getcwd()
        os.chdir(tmp)
        try:
            model = STEP(ds, os.path.join(tmp, "ts.pt"), ts_args(self.patches), gw_args(self.nodes),
                         dict(dataset_name=ds, k=10, input_seq_len=12, output_seq_len=12))
        finally:
            os.chdir(cwd)
        model.load_state_dict(dict(O.synthetic_trainable_params(ds, 0)), strict=False)
        model = model.to(dev).train()                 # the reference trains with the frozen TSFormer left in train()
        model.tsformer.chunk_seqs = chunk_seqs
        model.tsformer.precision = precision
        if no_dropout:
            model.tsformer.dropout_p = 0.0
            model.backend.dropout = 0.0
        self.model = model
        if mode == "node" and world > 1:
            # node-parallel: every rank holds the SAME batch, encodes its node range, one all-gather assembles the states;
            # everything after the gather is replicated and identical on every rank -> no gradient all-reduce
            model.tsformer.node_shard = (rank, world)
            self.reducer = parallel.GradReducer(model.parameters(), 1)
            seed_off = 0
        else:
            if os.environ.get("STEP_B200_REDUCER", "assign") == "flat":
                self.reducer = parallel.FlatGradReducer(model.parameters(), world)
            else:
                self.reducer = parallel.GradReducer(model.parameters(), world)
                self.overlap = world > 1 and os.environ.get("STEP_B200_OVERLAP_REDUCE", "1") != "0"
                if self.overlap:
                    model.discrete_graph_learning.before_trainable = self.reducer.wait
            seed_off = 17 * rank
        self.n_host = 4                               # rotate a few distinct host batches (inputs differ step to step)
        self.host = []
        for i in range(self.n_host):
            h, lh, f, _ = O.synthetic_batch(ds, batch, self.patches, 100 + seed_off + i)
            self.host.append((h.pin_memory(), lh.pin_memory(), f.pin_memory()))
        self.resident = [(h.to(dev), lh.to(dev), f.to(dev)) for (h, lh, f) in self.host[:2]]
        self.h2d_bytes = sum(t.numel() * 4 for t in self.host[0])

    def train_step(self, history, long_history, future):
        y_hat, theta, adj_knn, coeff = self.model(history_data=history, long_history_data=long_history, future_data=None,
                                                  batch_seen=0, epoch=1)
        loss = self.step_loss(y_hat[..., :1], future[..., :1], theta, adj_knn, coeff, null_val=0.0)
        # detached: holding the graph would keep the backward's saved tensors alive into the next step
        self.last_outputs = (y_hat.detach(), theta.detach(), adj_knn.detach(), coeff, loss.detach())
        self.reducer.zero()
        loss.backward()
        # NCCL all-reduce (big tensor in place + one packed buffer) when world > 1, enqueued on a side stream: it is joined
        # by the next step right after its frozen-encoder forward (discrete_graph_learning.before_trainable) and, for the
        # last timed step, by finish() inside the timed region
        self.reducer.reduce(async_op=self.overlap)
        return loss

    def finish(self):
        if self.overlap:
            self.reducer.wait()

    def samples_per_step(self):
        return self.B if (self.mode == "node") else self.B * self.world


def barrier(dev, world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize(dev)


def timed(fn, n, dev, world):
    barrier(dev, world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    barrier(dev, world)
    ms = e0.elapsed_time(e1)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return ms


def time_ms(fn, dev, reps=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def run_e2e(arm, steps, dev, world):
    """pinned host batch -> H2D copies -> step -> loss read back, all inside the timed region.  The copies of step i+1
    are issued on a side stream while step i computes (double-buffered device staging), the way a prefetching data
    loader feeds the runner; every byte is still copied inside the timed region and every step's loss is read back."""
    losses = []
    copy_stream = torch.cuda.Stream(dev)
    staging = [tuple(torch.empty_like(t, device=dev) for t in arm.host[0]) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def issue_copy(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])            # the step that last used this slot is done with it
            for dst, src in zip(staging[slot], arm.host[i % arm.n_host]):
                dst.copy_(src, non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_step(i):
        if i == 0:
            issue_copy(0)
        issue_copy(i + 1)                                       # prefetch the next batch during this step
        slot = i % 2
        torch.cuda.current_stream(dev).wait_event(ready[slot])
        loss = arm.train_step(*staging[slot])
        consumed[slot].record(torch.cuda.current_stream(dev))
        losses.append(loss.item())                              # D2H read of the step's result
        if i == steps - 1:
            arm.finish()
    for ev in consumed:
        ev.record(torch.cuda.current_stream(dev))
    e2e_step(0)
    torch.cuda.synchronize(dev)
    for ev in consumed:
        ev.record(torch.cuda.current_stream(dev))
    return timed(e2e_step, steps, dev, world), losses


def run_device_loader_leg(arm, steps, dev):
    """SURVEY section 8(f).1: the series stays resident on the GPU and every batch is gathered on the device from the window
    index (step.step_data.DeviceWindowLoader) - only the B sample indices cross PCIe, against 162 MB of overlapping host
    windows per METR-LA batch in the `e2e` leg.  Same step, loss read back every step."""
    from step.step_data import DeviceWindowLoader, ForecastingDataset
    ds = ForecastingDataset(synthetic=True, num_nodes=arm.nodes, seq_len=arm.patches * 12, length=arm.B * 8, seed=5)
    loader = DeviceWindowLoader(ds, dev, batch_size=arm.B, shuffle=True, drop_last=True, seed=1)
    batches = iter(())
    losses = []

    def step(i):
        nonlocal batches
        try:
            future, history, long_history = next(batches)
        except StopIteration:
            batches = iter(loader)
            future, history, long_history = next(batches)
        losses.append(arm.train_step(history, long_history, future).item())
    for i in range(3):
        step(i)
    ms = timed(step, steps, dev, 1)
    return {"value": arm.B * steps / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms / steps,
            "h2d_bytes_per_step": arm.B * 8, "d2h_bytes_per_step": 4,
            "what": "series resident in HBM (%.0f MB), windows gathered on the device per batch, loss read back every step"
                    % (ds.data.numel() * 4 / 1e6)}


def rooflines(arm, args, pk):
    """Kernels / kernel groups timed alone with CUDA events on the launching stream (after warm-up); algorithmic
    bytes / FLOPs per DESIGN.md section 4 (SURVEY section 8(d) and Appx B figures x the units one launch processes)."""
    from step_b200 import ops
    import torch.nn.functional as F
    dev, B, N, P, model = arm.dev, arm.B, arm.nodes, arm.patches, arm.model
    S_seq = B * N
    tokens = S_seq * P
    enc_flops = B * N * (4 * (P * (2 * 96 * 288 + 2 * 96 * 96 + 4 * 96 * 384) + 4 * 4 * P * P * 24) + 2 * P * 12 * 96)
    lh = arm.resident[0][1]
    shard = model.tsformer.node_shard
    model.tsformer.node_shard = None

    def enc_once():
        with torch.no_grad():
            return model.tsformer(lh[..., [0]])
    enc_ms = time_ms(enc_once, dev)
    enc_tflops = enc_flops / (enc_ms * 1e-3) / 1e12
    drop = 0.0 if args.no_dropout else 0.1
    other = [{"kernel": "TSFormer encoder, 21 launches (tc_embed + 4 x [QKV, attention, out+LN1, FFN1, FFN2+LN2])"
              if args.precision == "bf16" else "TSFormer encoder, fp32 CUDA-core kernels",
              "bound": "tensor", "achieved": enc_tflops, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
              "frac": enc_tflops / pk["bf16_tflops"], "ms": enc_ms, "useful_flops": enc_flops,
              "traffic": profile_traffic("r02_ncu_encoder_total.txt") if arm.ds == "METR-LA" and B == 32 and args.precision == "bf16" else None}]
    roofline = None
    if args.precision == "bf16":
        L = ops._L()
        x_img = ops.tc_rows_to_image(torch.randn(tokens, 96, device=dev))
        w_in = ops.tc_pack_weight(torch.randn(288, 96, device=dev) * 0.15)
        b_in = torch.zeros(288, device=dev)
        q = torch.empty(L.step_tc_attn_image_bytes(S_seq, P, 0), device=dev, dtype=torch.uint8)
        k = torch.empty(L.step_tc_attn_image_bytes(S_seq, P, 1), device=dev, dtype=torch.uint8)
        v = torch.empty(L.step_tc_attn_image_bytes(S_seq, P, 1), device=dev, dtype=torch.uint8)
        o = torch.empty(((tokens + 127) // 128) * 96 * 256, device=dev, dtype=torch.uint8)
        st = ops._enter(x_img)
        bound = torch.empty(L.step_tc_attn_image_bytes(S_seq, P, 2) // 4, device=dev, dtype=torch.float32)
        ops.check(L.step_tc_qkv(x_img.data_ptr(), w_in.data_ptr(), b_in.data_ptr(), S_seq, P, q.data_ptr(), k.data_ptr(),
                                v.data_ptr(), bound.data_ptr(), st), "step_tc_qkv")
        att_ms = time_ms(lambda: ops.check(L.step_tc_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                                              bound.data_ptr(), S_seq, P, drop, 1, st), "step_tc_attention"), dev)
        att_flops = 4.0 * S_seq * 4 * P * P * 24            # useful (unpadded) QK^T + PV flops of one layer
        att_tflops = att_flops / (att_ms * 1e-3) / 1e12
        w1 = ops.tc_pack_weight(torch.randn(384, 96, device=dev) * 0.1)
        b1 = torch.zeros(384, device=dev)
        ffn_ms = time_ms(lambda: ops.tc_linear(x_img, w1, b1, tokens, 96, 384, 1, drop_p=drop, seed=7), dev)
        ffn_bytes = tokens * (96 + 384) * 2.0                            # bf16 activations in + out (weights stay in smem)
        ffn_gbs = ffn_bytes / (ffn_ms * 1e-3) / 1e9
        prof = "r02_ncu_attn.txt" if os.path.exists(os.path.join(ROOT, "profiles", "r02_ncu_attn.txt")) else "r01_ncu_full_v5_attn.txt"
        roofline = {"kernel": "tc_attn_kernel<%d,%d> (one TSFormer layer: S=QK^T, softmax, PV on tcgen05; %d sequences x 4 heads, "
                              "P=%d, head dim 24)" % (P, 1 if drop > 0 else 0, S_seq, P),
                    "bound": "tensor", "achieved": att_tflops, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                    "frac": att_tflops / pk["bf16_tflops"], "ms": att_ms, "useful_flops": att_flops,
                    "traffic": profile_traffic(prof) if arm.ds == "METR-LA" and B == 32 else None,
                    "traffic_source": "profiles/%s (dram__bytes_read.sum + dram__bytes_write.sum per launch, parsed at run time; "
                                      "algorithmic q,k,v,o bf16 bytes = 855 MB)" % prof,
                    "peak_source": pk["source"] + " (burst cuBLAS bf16, kernel timed alone)",
                    "note": "head dim 24 makes this kernel exp/issue-bound, not MMA-bound (SURVEY section 7)"}
        other.append({"kernel": "tc_linear_kernel<1,0> (FFN1 [T,96]x[96,384] + bias + ReLU + dropout %.1f -> bf16 image), "
                                "timed with the dropout it runs with in the step" % drop, "bound": "hbm",
                      "achieved": ffn_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ffn_gbs / pk["hbm_gbs"],
                      "ms": ffn_ms, "algorithmic_bytes": ffn_bytes})
        del x_img, q, k, v, o
    else:
        roofline = dict(other[0])
        roofline["traffic"] = None
        roofline["peak_source"] = pk["source"]

    # ---- D4: cosine-similarity Gram (tcgen05, K = P*96) + global top-k: streams the bf16 sequence image once
    if args.precision == "bf16" and model.tsformer.seq_image is not None:
        img = model.tsformer.seq_image
        d4_ms = time_ms(lambda: ops.topk_mask(ops.tc_cosine_gram(img, B, N, P), 10 * N), dev)
        d4_bytes = B * N * P * 96 * 2.0 + B * N * N * 4.0            # bf16 states in, adjacency out
        other.append({"kernel": "D4 kNN prior: tc_gram_kernel + gram_normalize + topk_mask_kernel (3 launches)", "bound": "hbm",
                      "achieved": d4_bytes / (d4_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                      "frac": d4_bytes / (d4_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "ms": d4_ms, "algorithmic_bytes": d4_bytes,
                      "useful_flops": 2.0 * B * N * N * P * 96})

    # ---- D1: the batch-invariant trunk (conv1/bn1/conv2/bn2 kernels, fc + bn3 split-bf16 tcgen05 GEMMs), fwd + bwd
    dgl = model.discrete_graph_learning
    K = dgl.dim_fc

    def trunk_once():
        for p_ in dgl.parameters():
            p_.grad = None
        feat = dgl._global_feature(dev)
        feat.backward(torch.ones_like(feat))
    d1_ms = time_ms(trunk_once, dev, reps=5, warm=2)
    y2n = torch.randn(N, K, device=dev)
    fcw = [t.detach().clone().requires_grad_(True) for t in (dgl.fc.weight, dgl.fc.bias, dgl.bn3.weight, dgl.bn3.bias)]
    y2n.requires_grad_(True)

    def fc_once():
        y2n.grad = None
        for t in fcw:
            t.grad = None
        feat, _ = ops.TrunkFc.apply(y2n, *fcw, 1e-5, True, None, None)
        feat.backward(torch.ones_like(feat))
    fc_ms = time_ms(fc_once, dev, reps=5, warm=2)
    fc_bytes = 3.0 * (N + 100) * K * 4.0       # fwd reads X+W; bwd reads W, writes dX, reads X, writes dW
    other.append({"kernel": "D1 trunk fc + bn3 fwd+bwd: fc_fwd / fc_dx / fc_dw (split-bf16 tcgen05) + 4 small kernels", "bound": "hbm",
                  "achieved": fc_bytes / (fc_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                  "frac": fc_bytes / (fc_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "ms": fc_ms, "algorithmic_bytes": fc_bytes,
                  "useful_flops": 6.0 * N * 100 * K})
    L0 = dgl.train_length
    conv_flops = 3.0 * 2.0 * N * (8 * 10 * (L0 - 9) + 16 * 80 * (L0 - 18))
    other.append({"kernel": "D1 whole trunk fwd+bwd (conv1 / BatchNorm kernels, conv2 fwd+bwd as in-place implicit GEMMs on tcgen05, + the fc group above)", "bound": "hbm",
                  "achieved": (fc_bytes + 4.0 * N * 16 * (L0 - 18) * 4.0) / (d1_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"],
                  "unit": "GB/s", "frac": (fc_bytes + 4.0 * N * 16 * (L0 - 18) * 4.0) / (d1_ms * 1e-3) / 1e9 / pk["hbm_gbs"],
                  "ms": d1_ms, "algorithmic_bytes": fc_bytes + 4.0 * N * 16 * (L0 - 18) * 4.0,
                  "useful_flops": conv_flops + 6.0 * N * 100 * K,
                  "traffic": profile_traffic("r02_ncu_trunk_total.txt") if arm.ds == "METR-LA" else None,
                  "note": "conv trunk bytes = y2 and y2n written in forward, read in backward (y1 is recomputed)"})
    del y2n, fcw

    # ---- G2: the Graph WaveNet layer stack alone (north-star "diffusion-GCN + gated conv" path), HBM roofline
    gw = model.backend
    history = arm.resident[0][0]
    with torch.no_grad():
        x = F.pad(history[..., :2], (0, 0, 0, 0, 1, 0))
        x0 = (x @ gw.start_conv.weight.view(32, 2).t() + gw.start_conv.bias).contiguous()
        adj = (torch.rand(B, N, N, device=dev) < 0.5).float()
        adj.diagonal(dim1=1, dim2=2).zero_()
        P1, P2 = gw._random_walk(adj), gw._random_walk(adj.transpose(-1, -2))
        P3 = F.softmax(F.relu(gw.nodevec1 @ gw.nodevec2), dim=1)
    flat = gw._flat_layer_params()
    n_layers = gw.blocks * gw.layers

    def gw_fwd():
        with torch.no_grad():
            return ops.GWNetStack.apply(x0, P1, P2, P3, True, gw.dropout, 11, None, n_layers, *flat)
    gw_fwd_ms = time_ms(gw_fwd, dev)
    leaves = [t.detach().clone().requires_grad_(True) for t in (x0, P1, P2, P3)]
    dskip = torch.randn(B, N, 256, device=dev)

    def gw_fwdbwd():
        for t in leaves:
            t.grad = None
        for p_ in gw.parameters():
            p_.grad = None
        skip, _ = ops.GWNetStack.apply(*leaves, True, gw.dropout, 11, None, n_layers, *flat)
        skip.backward(dskip)
    gw_ms = time_ms(gw_fwdbwd, dev)
    act = 32.0 * N * 116 * 4 * B                        # x in + out of the 8 layers (SURVEY Appx B: 32*N*116*4 B per sample)
    sup = (2.0 * B + 1) * N * N * 4                     # dense fp32 supports (the sampled graph is ~50 % dense at init)
    stash = float(ops._L().step_gwnet_stash_floats(B, N, n_layers)) * 4
    skip_b = 2.0 * B * N * 256 * 4
    g2_fwd_bytes = act + sup + B * N * 256 * 4.0
    g2_all_bytes = 2 * act + 2 * sup + 2 * stash + skip_b
    other.append({"kernel": "G2 GWNet stack forward (step_gwnet_stack_fwd: one gw_fused_fwd_kernel per gcn layer [gated conv, both "
                            "diffusion hops on tcgen05, channel mixes, BN stats] + skip conv)", "bound": "hbm", "achieved": g2_fwd_bytes / (gw_fwd_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"],
                  "unit": "GB/s", "frac": g2_fwd_bytes / (gw_fwd_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "ms": gw_fwd_ms,
                  "algorithmic_bytes": g2_fwd_bytes,
                  "note": "algorithmic = layer inputs+outputs (32*N*116*4 B per sample) + dense supports + skip output; "
                          "the backward stash written here is NOT counted"})
    other.append({"kernel": "G2 GWNet stack forward + backward (stack_fwd + stack_bwd incl. dense dL/dP for the straight-through "
                            "estimator)", "bound": "hbm", "achieved": g2_all_bytes / (gw_ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"],
                  "unit": "GB/s", "frac": g2_all_bytes / (gw_ms * 1e-3) / 1e9 / pk["hbm_gbs"], "ms": gw_ms,
                  "algorithmic_bytes": g2_all_bytes, "stash_bytes": stash,
                  "traffic": profile_traffic("r02_ncu_gw_stack_total.txt") if arm.ds == "METR-LA" and B == 32 else None,
                  "note": "algorithmic = 2 x (activations + supports) + stash written and read once + skip in/out"})
    model.tsformer.node_shard = shard
    return roofline, other


def _claim_stdout():
    """Libraries print to stdout (NCCL's version banner does, whatever NCCL_DEBUG_FILE says): keep the real stdout for the
    ONE JSON line and point file descriptor 1 at stderr for everything else."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    args = parse()
    out_stream = _claim_stdout()
    ds = args.workload
    nodes, cfg_batch, patches = WORKLOADS[ds]
    if args.batch is None:
        args.batch = cfg_batch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and "NCCL_DEBUG" not in os.environ:
        # NCCL's own log (communicator size, rings, NVLS) goes to stderr: stdout carries only the JSON line
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

    if args.impl == "reference":
        if rank != 0:
            return
        b = 2 if (args.steps + args.warmup) <= 12 else 1
        v, info = cpu_reference_run(ds, args.steps, args.warmup, b)
        info["value"] = v
        print(json.dumps({"impl": "reference", "metric": metric_name(ds), "value": v, "unit": "samples/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * b / v,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
                          "data": "synthetic", "config": {"workload": "STEP_%s N=%d P=%d 12->12, CPU sample batch %d" % (ds, nodes, patches, b)},
                          "cpu_baseline": info,
                          "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), file=out_stream, flush=True)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200-native path has no CPU fallback "
                         "(use --impl reference for the CPU comparator)")
    import torch.distributed as dist
    from step_b200 import parallel
    from step_b200 import lib as _lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    parallel.init_from_env("nccl")
    torch.manual_seed(1234 + rank)

    arm = Arm(ds, args.batch, args.mode, args.precision, dev, rank, world, args.no_dropout, args.chunk_seqs)
    B = args.batch

    # ---- warm-up, then the device-resident measurement ----
    for i in range(max(args.warmup, 3)):
        arm.train_step(*arm.resident[i % 2])
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # kernels of libstep_b200.so enqueued inside the timed region, counted by the library itself (every launch site
    # goes through its check_launch); torch's own glue kernels are not included
    k0 = int(_lib.load().step_launch_count())
    def resident_step(i):
        arm.train_step(*arm.resident[i % 2])
        if i == args.steps - 1:
            arm.finish()
    ms_res = timed(resident_step, args.steps, dev, world)
    launches = int(_lib.load().step_launch_count()) - k0
    if args.dump_outputs and rank == 0:
        dump_outputs(arm, args.dump_outputs)
    if args.only_resident:
        if rank == 0:
            sampler.stop()
            print(json.dumps({"only_resident": True, "ms_per_step": ms_res / args.steps, "gpu_launches": launches}), file=out_stream, flush=True)
        return

    ms_e2e, losses = run_e2e(arm, args.steps, dev, world)
    clocks = sampler.stop() if rank == 0 else None

    pk = peaks()
    roofline, roofline_other = rooflines(arm, args, pk) if rank == 0 else (None, None)
    device_loader = run_device_loader_leg(arm, args.steps, dev) if world == 1 else None

    # ---- the other BASELINE configs, short runs (same timing rules; every rank takes part when they are multi-GPU) ----
    secondary = []
    if not args.no_secondary and ds == "METR-LA" and args.mode == "batch":
        del arm
        torch.cuda.empty_cache()
        plan = [("PEMS04", "batch")] if world == 1 else [("PEMS-BAY", "batch"), ("PEMS07", "node"), ("PEMS07", "batch")]
        for sds, smode in plan:
            try:
                a2 = Arm(sds, WORKLOADS[sds][1], smode, args.precision, dev, rank, world, args.no_dropout)
                for i in range(3):
                    a2.train_step(*a2.resident[i % 2])
                def sec_step(i, a2=a2):
                    a2.train_step(*a2.resident[i % 2])
                    if i == 4:
                        a2.finish()
                ms2 = timed(sec_step, 5, dev, world)
                secondary.append({"workload": "STEP_%s N=%d per-GPU batch %d P=%d" % (sds, a2.nodes, a2.B, a2.patches),
                                  "mode": smode, "n_gpus": world, "ms_per_step": ms2 / 5,
                                  "value": a2.samples_per_step() * 5 / (ms2 * 1e-3), "unit": "samples/s",
                                  "scaling": "strong (same batch on every rank, nodes sharded)" if smode == "node" and world > 1 else "weak",
                                  "steps": 5, "warmup": 3})
                del a2
                torch.cuda.empty_cache()
            except Exception as e:      # noqa: BLE001
                secondary.append({"workload": sds, "mode": smode, "error": repr(e)[:300]})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total_samples = (B if args.mode == "node" else B * world) * args.steps
    value = total_samples / (ms_res * 1e-3)
    e2e = total_samples / (ms_e2e * 1e-3)
    par = "single GPU"
    if world > 1:
        par = ("dp%d (batch-parallel, NCCL grad all-reduce)" % world if args.mode == "batch" else
               "node-parallel x%d (TSFormer sequences sharded by node, one NCCL all-gather of the states, rest replicated)" % world)
    out = {
        "metric": metric_name(ds), "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_res / args.steps, "higher_is_better": True,
        "scaling": "strong" if (args.mode == "node" and world > 1) else "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "fp32", "data": "synthetic",
        "config": {"workload": "STEP_%s fwd+loss+bwd, N=%d, per-GPU batch %d, P=%d (%d-step history), 12->12"
                               % (ds, nodes, B, patches, patches * 12),
                   "parallelism": par,
                   "dropout": "off" if args.no_dropout else "live (TSFormer 0.1 in train(), gcn 0.3) as the reference trains",
                   "l2": "inputs > L2: each step streams a fresh 160 MB long-history batch and ~1 GB of activations",
                   "precision": ("TSFormer encoder + Gram bf16 operands / fp32 accumulate on tcgen05; trunk Linear and GWNet node "
                                 "mixes split-bf16 (fp32-class) on tcgen05; everything else fp32"
                                 if args.precision == "bf16" else "fp32 everywhere"),
                   "ts_chunk_seqs": args.chunk_seqs,
                   "weights": ("real TSFormer_METR-LA encoder" if ds == "METR-LA" else "seeded random TSFormer encoder")
                              + ", seeded random GWNet/DGL"},
        "e2e": {"value": e2e, "unit": "samples/s", "h2d_bytes_per_step": arm_h2d(ds, B), "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline, "roofline_other": roofline_other,
        "loss": losses[-1] if losses else None,
    }
    if device_loader is not None:
        out["e2e_device_loader"] = device_loader
    if secondary:
        out["secondary"] = secondary
    if not args.no_eager_baseline and world == 1:
        out["gpu_eager_baseline"] = gpu_eager_baseline(ds, B, dev)
    if not args.no_cpu_baseline:
        v, info = cpu_reference_run(ds, 2, 1, 2)
        info["value"] = v
        info["unit"] = "samples/s"
        out["cpu_baseline"] = info
    print(json.dumps(out), file=out_stream, flush=True)
    if world > 1:
        dist.destroy_process_group()


def arm_h2d(ds, B):
    n, _, p = WORKLOADS[ds]
    return (2 * B * 12 * n * 3 + B * p * 12 * n * 3) * 4


if __name__ == "__main__":
    main()
