#!/usr/bin/env python3
"""bench.py — images/sec of the AlexNet (CLS_net_20140801232522) training step, one process per GPU.

    python bench.py --gpus N --steps K --warmup W              (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one synthetic batch: fprop, loss derivative, bprop
(wgrad + dgrad of every edge), the data-parallel gradient all-reduce (NCCL, N > 1) and the SGD
update, sequenced by the native host code (convnet_b200/host, the mirror of the reference's
ConvNet::TrainOneBatch) through the C ABI of libconvnet_b200.so.  Nothing is skipped: dropout,
bias, ReLU, softmax/CE and the optimizer run inside the timed region.

Prints ONE JSON line (rank 0).  `value` = images/s with the batch already resident in HBM;
`e2e` = the same step fed from pinned HOST buffers (H2D of images+labels and D2H of the loss inside
the timed region).  `--impl reference` times the reference's own CPU implementation of the same
step on the host cores (tools/cpu_reference.py) and prints the same line with "impl": "reference".

`--dump-outputs DIR` writes what the last resident timed step computed (rank 0) as DIR/<name>.npy, so that two
builds run with the same arguments, hence the same inputs, can be compared output for output (dump_outputs below).
The bench writes nothing into the source tree.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True                 # the tree may be read-only; keep it untouched either way
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"    # the CPU baseline's worker processes
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

METRIC = "images/sec ImageNet AlexNet training"
PER_GPU_BATCH = 128
WORKLOAD = ("examples/imagenet CLS_net_20140801232522 (AlexNet-style, 19 edges, 104.3 M params) training step, "
            "batch %d per GPU, synthetic 224x224x3" % PER_GPU_BATCH)


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx, self.windows = [], None, gpu_index, []

    def window(self, t0, t1):
        """a timed region [t0, t1] (time.time()): only samples taken inside a window are reported"""
        self.windows.append((t0, t1))

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        # nvidia-smi prints a sample a few ms after taking it: accept rows up to 30 ms past a window's end
        rows = [r for t, r in self.rows if any(a <= t <= b + 0.03 for a, b in self.windows)] if self.windows else \
               [r for _, r in self.rows]
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the step on the host cores (rank 0 only)."""
    if rank != 0:
        return
    import cpu_reference
    cores = os.cpu_count() or 1
    total = args.steps + args.warmup
    # every step is a bounded sample of the step's conv work; the whole run aims at <= ~3 minutes.  The layer set follows
    # from this budget alone (tools/cpu_reference.py), so the same command line always times the same layers
    per_step_budget = max(0.5, 160.0 / total)
    pool = cpu_reference.Pool(cores)
    vals, desc = [], ""
    t0 = time.perf_counter()
    for i in range(total):
        v, desc = pool.step(per_step_budget)
        if i >= args.warmup:
            vals.append(v)
    wall = time.perf_counter() - t0
    pool.close()
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * PER_GPU_BATCH / value,      # time of one batch-128 step at the measured rate (what `value` means)
        "sample_wall_ms_per_step": 1000.0 * wall / total, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "device": "host CPU", "sample_per_step": desc},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": pool.kind, "sample": desc},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def conv_roofline(torch, lib, peaks, peak_kind, iters=10):
    """the dominant kernel family of the step: tcgen05 implicit-GEMM conv.  Timed live (CUDA events on the
    launching stream) on the BASELINE headline layer: 3x3 conv fprop at batch 256 (conv4: 14x14x768 -> 384)."""
    from convnet_b200 import conv_gemm as cg
    from convnet_b200.abi import GetConvDesc
    from convnet_b200.matrix import CUDAMatrix
    N, W, Cin, Cout, k = 256, 14, 768, 384, 3
    d = GetConvDesc(Cin, Cout, k, k, 1, 1, 1, 1)
    x = CUDAMatrix(N, W * W * Cin, (N, W, W, Cin)); x.storage.normal_()
    w = CUDAMatrix(Cout, k * k * Cin, (Cout, k, k, Cin)); w.storage.normal_().mul_(0.02)
    y = CUDAMatrix(N, W * W * Cout, (N, W, W, Cout))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2
    L = lib.load()

    def timed_call(flush_l2=True):
        for _ in range(3):
            cg.convUp(x, w, y, d)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in ev:
            if flush_l2:
                flush.zero_()                                                # L2 flush between timed launches
            a.record(); cg.convUp(x, w, y, d); b.record()
        torch.cuda.synchronize()
        return statistics.median(a.elapsed_time(b) for a, b in ev)

    ms_warm = None
    ms_call = timed_call()                 # the plain ABI call: in bf16 mode it holds the two staging passes + the kernel
    path = lib.last_conv_path()
    ms = ms_call
    if path == "tcgen05-bf16":
        # what the training host does (EdgeWithWeight::StageForUp): operands staged once, the call is the kernel alone
        L.convnet_b200_bf16_stage(x.ptr, x.storage.numel())
        L.convnet_b200_bf16_stage(w.ptr, w.storage.numel())
        ms = timed_call()
        try:       # informational: back-to-back launches, no flush (the 159 MB working set already exceeds the 126 MB L2)
            ms_warm = timed_call(flush_l2=False)
        except Exception:
            ms_warm = None
        L.convnet_b200_bf16_invalidate(None)
    flops = 2.0 * N * W * W * Cout * k * k * Cin
    achieved = flops / (ms * 1e-3) / 1e12
    peak = peaks["bf16_tflops"]
    traffic = None                          # DRAM bytes per launch from the committed ncu --set full capture of this kernel
    if path == "tcgen05-bf16":
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_conv4_fprop_fast_ncu.json")))["traffic_bytes_per_launch"]
        except Exception:
            traffic = None
    return {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": traffic, "kernel": "tc_fast_kernel<fprop, pair> (%s)" % path,
            "shape": "conv4 fprop 3x3 s1 p1, 14x14x768 -> 384, batch 256 (266.3 GFLOP)", "ms_per_launch": ms,
            "back_to_back": None if not ms_warm else {"ms": ms_warm, "tflops": flops / (ms_warm * 1e-3) / 1e12,
                                                     "note": "same staged launch without the L2 flush between launches"},
            "unstaged_call": {"ms": ms_call, "tflops": flops / (ms_call * 1e-3) / 1e12,
                              "note": "same conv call with the fp32 -> bf16 staging passes of both operands inside it"},
            "peak_source": "%s bf16 burst peak (cuBLAS); %s" % (peak_kind, {
                "tcgen05-bf16": "bf16 operands staged beforehand (convnet_b200_bf16_stage, as the training step does), fp32 accumulate",
                "tcgen05-tf32": "the kernel multiplies in tf32, whose tensor peak is half of bf16"}.get(path, path))}


DUMP_SAMPLE = 1 << 22       # elements kept of a larger output: parameters and gradients are sampled (16 MB each)


def dump_outputs(torch, net, out_dir):
    """What the training step hands back, after the last timed step: the output layer's softmax probabilities, the summed
    cross-entropy of the batch, the updated parameters and their gradients.  Parameters and gradients are the same fixed,
    seeded sample of DUMP_SAMPLE positions inside the edges (never the padding between them); float32 .npy files."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    edges = [(off, size) for _, _, off, size in net.edges() if size > 0]
    offs, sizes = np.array([o for o, _ in edges], np.int64), np.array([s for _, s in edges], np.int64)
    starts = np.cumsum(sizes) - sizes
    total = int(sizes.sum())
    pick = np.unique(np.random.RandomState(0).randint(0, total, DUMP_SAMPLE)) if total > DUMP_SAMPLE else np.arange(total)
    e = np.searchsorted(starts, pick, side="right") - 1
    params = net.params_tensor()
    idx = torch.from_numpy(offs[e] + (pick - starts[e])).to(params.device)
    out = {"output": net.output_tensor().cpu().numpy(),
           "loss": np.array([net.loss()], np.float32),
           "params_sample": params[idx].cpu().numpy(),
           "grads_sample": net.grads_tensor()[idx].cpu().numpy()}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="alexnet")
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="images per GPU")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "tf32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true", help="e2e: copy each batch synchronously instead of one step ahead")
    ap.add_argument("--bucket-mb", type=float, default=128.0, help="gradient all-reduce bucket size")
    ap.add_argument("--no-cfg3", action="store_true", help="N > 1: skip the extra 256-images-per-GPU measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from convnet_b200 import lib
    from convnet_b200.net import Net, dp_unique_id

    torch.cuda.set_device(local_rank)
    L = lib.load()
    lib.set_precision(args.precision)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    net = Net(args.model, args.batch, seed=1234)         # identical initial parameters on every rank
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(dp_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        net.dp_init(rank, world, bytes(idt.cpu().numpy().tobytes()), int(args.bucket_mb * (1 << 20) / 4))

    # synthetic batch: N(0,1) pixels, uniform labels; seeds differ per rank like the reference (seed + rank)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    x_dev, y_dev = net.input_tensor(), net.labels_tensor()
    x_dev.normal_(generator=g)
    y_dev.copy_(torch.randint(0, net.num_classes, (args.batch,), device="cuda", generator=g, dtype=torch.int32))
    x_host = torch.empty(x_dev.numel(), dtype=torch.float32).pin_memory()
    y_host = torch.empty(args.batch, dtype=torch.int32).pin_memory()
    x_host.copy_(x_dev); y_host.copy_(y_dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)        # device time, max over ranks
        barrier()
        return ms.item()

    def step_resident():
        net.train_step(want_loss=False)                      # device-resident arm: no host round trip inside the loop

    losses = []

    # e2e input pipeline: the NEXT step's batch streams host -> device on a side stream into a staging buffer while the
    # current step computes (the reference's DataHandler prefetches the same way); every step still pays one full H2D of
    # its images + labels from pinned memory, one device copy into the net's input layer and one D2H of its loss.
    copy_stream = torch.cuda.Stream()
    x_stage, y_stage = torch.empty_like(x_dev), torch.empty_like(y_dev)
    ev_ready, ev_consumed = torch.cuda.Event(), torch.cuda.Event()

    def prefetch():
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_consumed)              # the previous step has read the staging buffer
            x_stage.copy_(x_host, non_blocking=True)         # H2D of the next step's images + labels from pinned memory
            y_stage.copy_(y_host, non_blocking=True)
            ev_ready.record(copy_stream)

    def step_e2e():
        torch.cuda.current_stream().wait_event(ev_ready)
        x_dev.copy_(x_stage); y_dev.copy_(y_stage)           # staging -> the net's input layer (device copy, compute stream)
        ev_consumed.record()
        if not args.no_prefetch:
            prefetch()
        losses.append(net.train_step(want_loss=True))        # D2H of the step's loss
        if args.no_prefetch:
            prefetch(); copy_stream.synchronize()            # serial variant: the copy is not overlapped with compute

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                      # nvidia-smi needs ~1 s to deliver its first sample
    for _ in range(args.warmup):
        step_resident()
    L.convnet_b200_reset_launch_count()
    t0 = time.time()
    ms_total = timed(step_resident, args.steps)
    sampler.window(t0, time.time())
    launches = int(L.convnet_b200_launch_count())
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, net, args.dump_outputs)
    ev_consumed.record()
    prefetch()                                               # the first timed step's batch
    for _ in range(2):
        step_e2e()
    t0 = time.time()
    ms_e2e = timed(step_e2e, args.steps)
    sampler.window(t0, time.time())                          # both timed regions run the same step under load
    clocks = sampler.stop() if rank == 0 else None

    # replicas must still be in lock-step after the timed loops: a 64-bit checksum of the raw parameter bits, compared
    # across ranks (the all-reduce result is identical on every rank, so every replica applied the same update)
    p_bits = net.params_tensor().view(torch.int32).to(torch.int64)
    checksum = (p_bits * (torch.arange(p_bits.numel(), device="cuda", dtype=torch.int64) % 8191 + 1)).sum().reshape(1)
    replicas_identical = True
    if world > 1:
        sums = [torch.zeros_like(checksum) for _ in range(world)]
        dist.all_gather(sums, checksum)
        replicas_identical = all(int(t.item()) == int(sums[0].item()) for t in sums)
        assert replicas_identical, "parameters diverged across ranks: %s" % [int(t.item()) for t in sums]

    # where the step's time goes on this rank: one traced step after the timed region (not part of any reported rate)
    timeline = net.trace_step()

    # BASELINE config 3 quotes the data-parallel run at 256 images per GPU: a second, shorter measurement of the same step at
    # that per-GPU batch (same net, same NCCL path), reported inside `config` — the headline stays config 2's batch 128
    cfg3 = None
    if world > 1 and not args.no_cfg3 and args.batch != 256:
        net3 = Net(args.model, 256, seed=1234)
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(dp_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        net3.dp_init(rank, world, bytes(idt.cpu().numpy().tobytes()), int(args.bucket_mb * (1 << 20) / 4))
        net3.input_tensor().normal_(generator=g)
        net3.labels_tensor().copy_(torch.randint(0, net3.num_classes, (256,), device="cuda", generator=g, dtype=torch.int32))
        for _ in range(3):
            net3.train_step(want_loss=False)
        steps3 = max(5, args.steps // 3)
        ms3 = timed(lambda: net3.train_step(want_loss=False), steps3)
        cfg3 = {"per_gpu_batch": 256, "images_per_s": 256 * world * steps3 / (ms3 * 1e-3), "ms_per_step": ms3 / steps3, "steps": steps3}
        net3.close()

    images = args.batch * world * args.steps
    value = images / (ms_total * 1e-3)
    e2e_value = images / (ms_e2e * 1e-3)

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        roof = conv_roofline(torch, lib, peaks, peak_kind)
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"tf32": "tf32", "bf16": "bf16", "fp32": "f32"}[args.precision], "data": "synthetic",
            "config": {"workload": WORKLOAD if args.model == "alexnet" else args.model, "global_batch": args.batch * world,
                       "per_gpu_batch": args.batch, "parallelism": "dp%d" % world,
                       "arithmetic": "fp32 storage and master weights; conv/1x1/fc multiply in %s on tcgen05 with fp32 accumulate "
                                     "(conv1, Cin=3, always tf32); pool/rnorm/elementwise fp32" % args.precision,
                       "l2": "no flush needed: one step streams >3 GB of activations/weights through the 126 MB L2",
                       "sync": ("NCCL all-reduce(avg) of the flat gradient buffer in buckets of >= %.0f MB cut at layer boundaries, on "
                                "its own stream as soon as a bucket's last wgrad is done, each followed by that bucket's SGD step on the "
                                "optimizer stream; NCCL width %s CTAs = SMs the conv grids leave free meanwhile"
                                % (args.bucket_mb, os.environ.get("CONVNET_B200_NCCL_CTAS", "16" if world <= 4 else "24")))
                               if world > 1 else "single GPU",
                       "train_gflop_per_image": net.flops_train / args.batch / 1e9,
                       "baseline_config3_256_per_gpu": cfg3},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(x_host.numel() * 4 + y_host.numel() * 4), "d2h_bytes_per_step": 4,
                    "pipeline": "serial H2D" if args.no_prefetch else "H2D of step i+1 on a side stream during step i"},
            "gpu_launches": launches,
            "model_tflops": value * net.flops_train / args.batch / 1e12,
            "roofline": roof,
            "last_loss": losses[-1] if losses else None,
            "param_checksum": int(checksum.item()), "replicas_identical": replicas_identical,
            "timeline_rank0": timeline,
        }
        if world == 1 and not args.no_cpu_baseline:
            import cpu_reference
            line["cpu_baseline"] = cpu_reference.measure(25.0)
        print(json.dumps(line), flush=True)
    net.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
