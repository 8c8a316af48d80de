#!/usr/bin/env python
"""bench.py -- CycleGAN-VC training-step throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16x3|bf16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the hot path over one synthetic minibatch: G_A2B/G_B2A/D_A/D_B forward + cycle/identity/
adversarial losses + backward + both Adam updates on batch 256 x [24 MCEP, 128 frames] per GPU (BASELINE.json
configs[2]/[3]; weak scaling: every GPU gets its own 256 samples, one NCCL all-reduce of the 479 MB gradient arena).

Prints ONE JSON line (rank 0).  `value` is 256-sample steps per second summed over all GPUs, timed with CUDA events
on device-resident inputs; `e2e` is the same through CycleGAN.train() with host buffers (H2D of A and B and D2H of
the losses inside the timed region).  `--impl reference` times the CPU oracle (a torch-CPU restatement of the
reference graph; TensorFlow 1.x cannot be installed here -- see DESIGN.md) on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step computed, as float32 `.npy` files, so that two builds can be compared
output for output (inputs and initial weights are seeded, so the same arguments give the same inputs in every run):
  train: losses.npy (the 8 losses, cgvc.native.LOSS_NAMES order) and params_sample.npy (the updated weights at DUMP_SAMPLE
         positions of the parameters concatenated in CycleGAN.param_names() order, drawn without replacement with seed 0, ascending);
  infer: converted_A2B.npy (the whole [1024, 24, 128] generator output).
The generator forward is deterministic: two runs of one build give bit-identical infer dumps.  A train step is not (the order of
its gradient atomics varies, and Adam's sign-descent early steps amplify that), so two runs of one build differ too: measured
after 3 warm-up + 10 timed default steps on a B200 at a 1000 W power limit, 7e-4 relative L2 on losses.npy and 5e-3 on
params_sample.npy.  Compare train dumps of two builds against that spread, not for equality.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (which may be read-only)

BATCH = 256
FRAMES = 128
FEATS = 24
LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D = 10.0, 5.0, 2e-4, 1e-4     # train.py:17-26
GFLOP_PER_SAMPLE_STEP = 91.41                                   # SURVEY.md section 8(d): conv FLOPs of the reference's graph (D(fake) run twice)
GFLOP_EXECUTED_PER_SAMPLE_STEP = 85.96                          # what the engine executes (D(fake) forward shared; DESIGN.md section 4)
GFLOP_GENERATOR_FWD = 2.656043                                  # one generator application per sample (T = 128)
METRIC = "CycleGAN-VC train steps/sec @ batch 256x[24,128] MCEP"
UNIT = "steps/s (256-sample steps, summed over GPUs)"
DUMP_SAMPLE = 1 << 22                                           # weights in params_sample.npy (16 MB of the 479 MB)


def dump_train_outputs(m, losses, out_dir):
    """--dump-outputs of the train workload: the last step's losses and a fixed sample of the weights it left."""
    import numpy as np
    flat = np.concatenate([p.ravel() for p in m.get_params().values()])
    pick = np.sort(np.random.default_rng(0).choice(flat.size, DUMP_SAMPLE, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "losses.npy"), np.asarray(losses, dtype=np.float32))
    np.save(os.path.join(out_dir, "params_sample.npy"), flat[pick])


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def _ncu_traffic(kernel_class):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture (profiles/*ncu_tc_kernels_summary.json; average over the captured launches), or None."""
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_tc_kernels_summary.json")),
                   key=lambda f: [int(x) for x in re.findall(r"\d+", os.path.basename(f))])      # r01_v10 after r01_v7
    if not files:
        return None
    try:
        d = json.load(open(files[-1]))
        ks = d["prof_tn" if kernel_class == 1 else "prof_nt"]
        vals = [(k["dram_read_MB"] + k["dram_write_MB"]) * 1e6 for k in ks if k.get("dram_read_MB") is not None]
        return sum(vals) / len(vals) if vals else None
    except Exception:
        return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


_SAVED_STDOUT = None


def mute_stdout():
    """NCCL prints a "NCCL version ..." banner on fd 1 when a communicator is created; rank 0's stdout must carry the JSON line only.
    Point fd 1 at stderr for the duration of the run; emit() restores it for the one line."""
    global _SAVED_STDOUT
    if _SAVED_STDOUT is None:
        sys.stdout.flush()
        _SAVED_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    global _SAVED_STDOUT
    sys.stdout.flush()
    if _SAVED_STDOUT is not None:
        os.dup2(_SAVED_STDOUT, 1); os.close(_SAVED_STDOUT); _SAVED_STDOUT = None
    print(json.dumps(line), flush=True)


def usable_cores():
    """Host cores this process may really use: min(affinity, cgroup cpu quota).  (The GPU boxes expose 128 logical CPUs
    but cap the container at a quota; oversubscribing torch's thread pool past the quota is catastrophically slow.)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, n)


def _cpu_model_name():
    try:
        return [l.split(":")[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        return "unknown"


def cpu_generator_forward_ms(threads, reps=5):
    """BASELINE.json configs[0]: generator_gatedcnn forward on random fp32 MCEP [1,24,128] on the CPU restatement (median of `reps`)."""
    import torch
    from oracle import cyclegan_oracle as O
    torch.set_num_threads(threads)
    P = O.init_params(seed=0, dtype=torch.float32)
    x, _ = O.synthetic_batch(0, 1, FRAMES)
    ts = []
    with torch.no_grad():
        O.generator_forward(x, P, "generator_A2B")
        for _ in range(reps):
            t0 = time.perf_counter(); O.generator_forward(x, P, "generator_A2B"); ts.append(time.perf_counter() - t0)
    return 1e3 * statistics.median(ts)


def cpu_reference_arm(steps, warmup, sample_batch, threads=None, with_config1=True):
    """The reference's CPU path, restated (oracle/cyclegan_oracle.py): `steps` full train steps (6 generator + 6 discriminator
    passes, autograd, TF Adam) on `sample_batch` samples each, after `warmup` untimed ones."""
    import torch
    from oracle import cyclegan_oracle as O
    cores = threads or usable_cores()
    torch.set_num_threads(cores)
    m = O.OracleCycleGAN(dtype=torch.float32, seed=0)
    A, B = O.synthetic_batch(0, sample_batch, FRAMES)
    A, B = A.numpy(), B.numpy()
    for _ in range(warmup):
        m.train(A, B, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    t0 = time.perf_counter()
    for _ in range(steps):
        m.train(A, B, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    value = (sample_batch / BATCH) / dt          # 256-sample steps per second
    out = {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "batch_per_step": sample_batch, "steps": steps, "warmup": warmup,
           "sec_per_step": dt, "sec_per_sample": dt / sample_batch, "cpu": _cpu_model_name(),
           "sample": ("%d timed full train steps on a minibatch of %d x [24,128] (after %d warm-up), %.2f s per step; " % (steps, sample_batch, warmup, dt))
                     + ("the whole batch-256 workload, measured" if sample_batch == BATCH else
                        "value = (%d/256 of a 256-sample step) / measured step time" % sample_batch)
                     + "; oracle = torch-CPU fp32 restatement of the TF1 graph (TF 1.x not installable, DESIGN.md section 9)"}
    if with_config1:
        out["generator_forward_1x24x128_ms"] = cpu_generator_forward_ms(cores)      # BASELINE.json configs[0]
    return out


def pick_reference_batch(steps, warmup, budget_s, threads):
    """Largest minibatch in {256, 128, 64, 32, 16} whose (steps + warmup) CPU train steps fit the time budget, from a batch-4 probe."""
    import torch
    from oracle import cyclegan_oracle as O
    torch.set_num_threads(threads)
    m = O.OracleCycleGAN(dtype=torch.float32, seed=0)
    A, B = O.synthetic_batch(1, 4, FRAMES)
    m.train(A.numpy(), B.numpy(), LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    t0 = time.perf_counter()
    m.train(A.numpy(), B.numpy(), LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    per_sample = (time.perf_counter() - t0) / 4.0
    for b in (256, 128, 64, 32, 16):
        if (steps + warmup) * b * per_sample <= budget_s:
            return b, per_sample
    return 16, per_sample


def infer_measure(precision, local_rank, world, dist, steps, warmup, dump_dir=None):
    """BASELINE.json configs[4] (convert.py path): generator-only A2B forward of 1024 x [24,128] per GPU.  Embarrassingly parallel
    over GPUs (no collective).  Returns a dict (rank 0) with frames/s device-resident and end to end (host numpy in / out).
    With `dump_dir`, the output of the last timed forward goes to dump_dir/converted_A2B.npy."""
    import numpy as np
    import torch
    import cgvc
    dev = torch.device("cuda", local_rank)
    nb = 1024
    m = cgvc.CycleGAN(num_features=FEATS, mode="test", max_batch=nb, max_frames=FRAMES, precision=precision, device=local_rank, seed=0)
    g = torch.Generator(device=dev); g.manual_seed(2000)
    x = torch.randn(nb, FEATS, FRAMES, device=dev, generator=g)
    for _ in range(max(warmup, 3)):
        m.test(x, "A2B")
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        y = m.test(x, "A2B")
    e1.record(); torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    if dump_dir is not None:
        os.makedirs(dump_dir, exist_ok=True)
        np.save(os.path.join(dump_dir, "converted_A2B.npy"), y.cpu().numpy())
    # end to end: host float32 utterance crops in, converted host array out (pinned staging, H2D + D2H inside the timed region)
    xh = x.cpu().numpy()
    m.test(xh, "A2B")
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e_steps = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(e_steps):
        yh = m.test(xh, "A2B")
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([ms, e2e_s], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms, e2e_s = float(t[0].item()), float(t[1].item())
    del m
    torch.cuda.empty_cache()
    fps = world * nb * FRAMES * steps / (ms / 1e3)
    tfl = world * nb * GFLOP_GENERATOR_FWD * 1e-3 * steps / (ms / 1e3)
    pk = _peaks()
    return {"metric": "convert.py A2B generator forward, batch 1024x[24,128]", "value": fps, "unit": "frames/s (summed over GPUs)",
            "n_gpus": world, "steps": steps, "ms_per_step": ms / steps, "dtype": precision, "tflops": tfl,
            "roofline": {"bound": "tensor", "achieved": tfl / world, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s per GPU",
                         "frac": tfl / world / pk["bf16_tflops_sustained"],
                         "note": "algorithmic conv FLOPs (2.656 GF per sample) / whole-forward time, of %s sustained bf16 peak" % pk["src"]},
            "e2e": {"value": world * nb * FRAMES * e_steps / e2e_s, "unit": "frames/s (summed over GPUs)", "steps": e_steps,
                    "h2d_bytes_per_step": int(xh.nbytes), "d2h_bytes_per_step": int(yh.nbytes)}}


def infer_bench(args, rank, local_rank, world):
    import torch
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    r = infer_measure(args.precision, local_rank, world, dist, args.steps, args.warmup, dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        r.update({"warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic", "clocks": clocks,
                  "config": {"workload": "generator_gatedcnn forward 1024 x [24,128] per GPU (BASELINE config 5)", "precision": args.precision,
                             "parallelism": "replicas x%d, no collective" % world}})
        emit(r)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="f16f8", choices=["f16f8", "bf16x3", "bf16", "fp32"],
                    help="f16f8 (default) and bf16x3 are the two parity-grade tensor-core precisions (2 and 3 MMA units per product)")
    ap.add_argument("--batch", type=int, default=BATCH, help="per-GPU minibatch (the metric is quoted at 256)")
    ap.add_argument("--cuda-graph", type=int, default=1, choices=[0, 1], help="replay the step as CUDA graphs (engine default) or launch eagerly")
    ap.add_argument("--fuse-bwd", type=int, default=-1, choices=[-1, 0, 1],
                    help="GLU/instance-norm backward fused into the data-gradient epilogue (residual stack): -1 = engine default")
    ap.add_argument("--cpu-sample-batch", type=int, default=0,
                    help="minibatch of the CPU legs: 0 = automatic (reference arm: the largest of 256/128/64/32/16 whose steps + warm-up fit "
                         "--cpu-budget-s; cpu_baseline of our arm: 32)")
    ap.add_argument("--cpu-budget-s", type=float, default=900.0, help="time budget of the `--impl reference` run")
    ap.add_argument("--no-infer", action="store_true", help="skip the BASELINE config-5 (generator-only inference) measurement added to the line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--replicas-only", action="store_true",
                    help="diagnostic for N > 1: every rank trains its own replica with no gradient exchange (what the step costs without the all-reduce, timed as the max over ranks like the real run); the line is marked and is not a data-parallel result")
    ap.add_argument("--set-option", action="append", default=[], metavar="NAME=VALUE",
                    help="engine option (include/cgvc.h: side_wgrad, cta_pairs, post_onepass, fuse_in, ...) for A/B measurements; repeatable")
    ap.add_argument("--workload", default="train", choices=["train", "infer"],
                    help="train: the headline metric; infer: BASELINE config 5, generator-only forward of 1024 x [24,128] (frames/s)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/*.npy (float32; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs records the native engine's outputs (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        mute_stdout()
    steps, warmup = args.steps, max(args.warmup, 3 if args.impl == "ours" else 0)
    workload = ("full CycleGAN-VC train step (4 generator + 2 discriminator applications fwd, losses, bwd, 2x Adam), "
                "batch %d x [24 MCEP, 128 frames] per GPU, synthetic N(0,1) MCEP, glorot weights" % args.batch)
    config = {"workload": workload, "per_gpu_batch": args.batch, "frames": FRAMES, "parallelism": "dp%d" % max(world, 1), "precision": args.precision,
              "l2": "per-step working set ~12 GB of activations >> 126 MB L2, no flush needed",
              "launch": "cuda_graph" if args.cuda_graph else "eager"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # every step = one full CPU train step on a minibatch sized so that warm-up + steps fit the budget; K and W are honoured
        cores = usable_cores()
        r_steps, r_warm = steps, max(args.warmup, 0)
        if args.cpu_sample_batch > 0:
            nb, probe = args.cpu_sample_batch, None
        else:
            nb, probe = pick_reference_batch(r_steps, r_warm, args.cpu_budget_s, cores)
        cb = cpu_reference_arm(steps=r_steps, warmup=r_warm, sample_batch=nb, threads=cores)
        if probe is not None:
            cb["batch_choice"] = "batch-4 probe: %.3f s per sample -> batch %d for %d + %d steps within %.0f s" % (probe, nb, r_steps, r_warm, args.cpu_budget_s)
        rcfg = {"workload": workload, "per_gpu_batch": args.batch, "frames": FRAMES, "parallelism": "cpu x%d threads" % cores,
                "measured_batch_per_step": nb, "implementation": "oracle/cyclegan_oracle.py (torch-CPU fp32 restatement of the TF1 graph)"}
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": 0, "steps": r_steps, "warmup": r_warm,
                "ms_per_step": 1e3 * cb["sec_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": rcfg, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
                "model_gflops": (nb * GFLOP_PER_SAMPLE_STEP) / cb["sec_per_step"]}
        emit(line)
        return 0

    import numpy as np
    import torch
    import cgvc
    from cgvc import native
    import ctypes as C

    if args.workload == "infer":
        return infer_bench(args, rank, local_rank, world)
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    m = cgvc.CycleGAN(num_features=FEATS, mode="train", max_batch=args.batch, max_frames=FRAMES, precision=args.precision,
                      device=local_rank, seed=0, data_parallel=world > 1 and not args.replicas_only, log_dir="/tmp/cgvc_bench_log")
    if args.replicas_only:
        config["replicas_only"] = True
    lib = native.load()
    lib.cgvc_set_option(m._handle, b"cuda_graph", args.cuda_graph)
    if args.fuse_bwd >= 0:
        lib.cgvc_set_option(m._handle, b"fuse_bwd", args.fuse_bwd)
        config["fuse_bwd"] = args.fuse_bwd
    wgrad_f16 = 1 if args.precision == "f16f8" else 0              # the engine's default in that precision (include/cgvc.h)
    for kv in args.set_option:
        name, value = kv.split("=")
        m.set_option(name, int(value))
        config.setdefault("options", {})[name] = int(value)
        if name == "wgrad_f16" and args.precision == "f16f8":
            wgrad_f16 = int(value)
    if args.precision == "f16f8":
        config["mma_units_per_product"] = {"forward": 2, "data_gradient": 2, "weight_gradient": 1 if wgrad_f16 else 2}
    g = torch.Generator(device=dev); g.manual_seed(1000 + rank)
    A = torch.randn(args.batch, FEATS, FRAMES, device=dev, generator=g)
    B = torch.randn(args.batch, FEATS, FRAMES, device=dev, generator=g)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        m.train_async(A, B, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = C.c_ulonglong(0); lib.cgvc_kernel_launches(C.byref(n0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        m.train_async(A, B, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    n1 = C.c_ulonglong(0); lib.cgvc_kernel_launches(C.byref(n1))
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    ms_per_step = ms / steps
    value = world * (args.batch / BATCH) * steps / (ms / 1e3)
    losses = m._losses.cpu().numpy().tolist()
    if args.dump_outputs is not None and rank == 0:
        dump_train_outputs(m, losses, args.dump_outputs)            # before the untimed steps below move the weights on

    # ---- end to end through the reference-facing API: host numpy in, losses out, copies inside the timed region
    A_host = A.cpu().numpy().astype(np.float32); B_host = B.cpu().numpy().astype(np.float32)
    for _ in range(2):
        m.train(A_host, B_host, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
    barrier()
    e_steps = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(e_steps):
        m.train(A_host, B_host, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)      # H2D of A and B, D2H of the 8 losses, stream sync
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t.item())
    e2e = {"value": world * (args.batch / BATCH) * e_steps / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": int(A_host.nbytes + B_host.nbytes), "d2h_bytes_per_step": 32, "steps": e_steps}

    # ---- roofline of the dominant kernel: per-launch CUDA-event timing of the tensor-core gather-GEMM kernels
    roofline = None
    if args.precision != "fp32":
        # per-launch timing needs the kernels of the two lanes serialised: one stream for this pass (2 untimed + 2 recorded steps)
        lib.cgvc_set_option(m._handle, b"two_streams", 0)
        for _ in range(2):
            m.train_async(A, B, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
        torch.cuda.synchronize(dev)
        lib.cgvc_profile_enable(1)
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        for _ in range(2):
            m.train_async(A, B, LAMBDA_CYCLE, LAMBDA_ID, LR_G, LR_D)
        pe1.record()
        ms2 = (C.c_double * 3)(); fl2 = (C.c_double * 3)(); ln2 = (C.c_longlong * 3)()
        lib.cgvc_profile_collect(ms2, fl2, ln2)
        lib.cgvc_profile_enable(0)
        lib.cgvc_set_option(m._handle, b"two_streams", 1)
        ms_per_step_1stream = pe0.elapsed_time(pe1) / 2.0
        pk = _peaks()
        k = max(range(3), key=lambda i: ms2[i])            # the dominant kernel class of the step
        knames = ["tc_pair_nt_kernel<BN,NPL,0> (conv forward + data-gradient gather-GEMM on CTA pairs, TMA im2col operand; the 15-tap 24-channel edge layers run as dense 1 x 1 layers on the same kernel)",
                  "tc_pair_tn_kernel / tc_pair_tn_q_kernel (weight-gradient gather-GEMM on CTA pairs; tc_gg_tn_kernel where a layer has < 256 channels or columns)",
                  "tc_pair_nt_kernel<256,NPL,1|2> (conv forward with the fused instance-norm + GLU / + residual epilogue)"]
        if ln2[k] > 0 and ms2[k] > 0:
            achieved = fl2[k] / (ms2[k] * 1e-3) / 1e12
            peak = pk["bf16_tflops_sustained"]
            roofline = {"bound": "tensor", "kernel": knames[k],
                        "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": _ncu_traffic(k),
                        "note": "achieved = algorithmic conv FLOPs (2*M*N*K, counted once) / summed CUDA-event time of %d launches over 2 steps (%.3f ms per launch avg); "
                                "peak = %s sustained dense bf16 (cuBLAS); each product costs 3 bf16 MMAs in bf16x3 mode (frac bounded by 1/3) and 2 MMA units in f16f8 mode (one fp16 MMA + two e4m3 MMAs at twice the rate: bounded by 1/2; the weight-gradient kernel of that mode issues the fp16 MMA alone unless wgrad_f16=0); mma_rate_frac = issued MMA units / peak; "
                                "timed with the two lanes of the step serialised on one stream; traffic = mean DRAM bytes (read + write) per launch over the launches of this kernel in the newest committed ncu --set full capture "
                                "(profiles/*ncu_tc_kernels_summary.json, newest version; the file lists the launches it holds)"
                                % (ln2[k], ms2[k] / ln2[k], pk["src"]),
                        "mma_rate_frac": achieved * {"bf16x3": 3.0, "f16f8": 2.0}.get(args.precision, 1.0) / peak,
                        # operand bytes the kernel pulls from L2 into shared memory: (128 + 256) rows x K x 4 B per 128 x 256 tile
                        # (two 2-byte planes per operand) = 0.0234 B per algorithmic FLOP; the L2 slice throughput cap of this chip
                        # (~6300 B/clk, B300_MICROARCH.md) is ~12 TB/s -- the ceiling the long-K layers sit at (DESIGN.md section 7)
                        "l2_operand_tbs": achieved * 0.0234375 if args.precision != "bf16" else achieved * 0.0234375 / 2,
                        "share_of_step": ms2[k] / 2.0 / ms_per_step_1stream, "ms_per_step_single_stream": ms_per_step_1stream,
                        "other_kernels": [{"kernel": knames[i], "ms_per_step": ms2[i] / 2.0,
                                           "tflops": (fl2[i] / (ms2[i] * 1e-3) / 1e12) if ms2[i] > 0 else None} for i in range(3) if i != k]}

    # ---- BASELINE config 5 beside the headline: generator-only forward of 1024 x [24,128] per GPU (convert.py path), every rank its own
    infer = None
    if not args.no_infer:
        infer = infer_measure(args.precision, local_rank, world, dist, steps=max(3, min(steps, 10)), warmup=3)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    cb = None
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_arm(steps=1, warmup=1, sample_batch=args.cpu_sample_batch or 32)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16x3": "bf16x3 (3 bf16 MMAs per product, f32 accumulate)", "bf16": "bf16", "fp32": "f32",
                      "f16f8": "f16f8 (forward / data gradient: fp16 MMA + two e4m3 cross-term MMAs = 2 MMA units per product; weight gradient: "
                               + ("fp16 MMA alone, 1 unit" if wgrad_f16 else "the same 2 units") + "; f32 accumulate)"}[args.precision],
            "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(n1.value - n0.value),
            "roofline": roofline, "cpu_baseline": cb,
            # conv FLOPs only: the reference's graph runs D(fake) twice (91.41 GF/sample); the engine shares that forward (85.96 GF/sample)
            "model_tflops_reference_graph": world * args.batch * GFLOP_PER_SAMPLE_STEP * 1e-3 * steps / (ms / 1e3),
            "executed_tflops": world * args.batch * GFLOP_EXECUTED_PER_SAMPLE_STEP * 1e-3 * steps / (ms / 1e3),
            "infer": infer,
            "losses_last_step": dict(zip(native.LOSS_NAMES, losses))}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
