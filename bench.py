"""Headline benchmark: MNIST MLP samples/sec, sync-replica parameter server, device-timed, max over ranks.

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` (N>1: launched with
``python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...``).  Rank 0 prints ONE
JSON line.  Config named by BASELINE.json: between-graph parameter server, 784-100-10 MLP, batch 100
per worker, clipped batch-sum cross-entropy, sync replicas (``replicas_to_aggregate = num_workers``),
fp32 storage with TF32 tensor-core multiplies (the reference model is fp32; ``--precision bf16`` = config 3).
Topology: every listed worker trains (/root/reference/distributed_mnist.py:27-29,120-122): N GPUs = N workers,
ps shard s shares worker s's GPU; ``--ps-only-task 1`` gives the ps its own GPU (1 ps + (N-1) workers).

* ``value``: whole-job samples/sec.  The timed region is EXACTLY K steps, run as ``reps`` equal repetitions (up to 10, each
  at least 100 steps when K allows; one CUDA-graph replay chain each) between CUDA events on every rank's stream, after a
  barrier + synchronize and two untimed alignment steps; MAX over ranks per repetition; the MEDIAN repetition is reported.
  The step count does not depend on timing, so a run with the same arguments computes the same steps.
* ``--dump-outputs DIR``: after the timed steps, what they computed -- the loss of the last step, the parameters and optimizer
  slots a caller would read back (``PSTrainEngine.state_dict``) -- as ``DIR/<name>.npy`` (float32 / float64, <= 64 MB in all),
  so that two builds can be compared output for output.
* inputs: a 55 000 x 784 fp32 synthetic MNIST-shaped training set resident in each worker's HBM
  (172 MB > the 126 MB L2), batches walked in order; the step kernel's TMA reads them in place.
* ``e2e``: the same metric through the public API with, every step, the host->device copy of that step's batch from pinned host
  memory and a device->host read of the loss (same repetition protocol).  Three arms, the best one reported, all kept:
  ``synchronous`` (``PSTrainEngine.step(x, y) -> loss``), ``pipelined`` (``step(..., sync_loss="deferred")``: the loss read one
  step late) and ``native_loop`` (``PSTrainEngine.train_loop(batches, steps=K)``: the K steps enqueued by one native call).
* ``vs_baseline``: value / the in-repo torch + NCCL + cuBLAS (CUDA-graphed) arm measured in the SAME invocation with the
  same steps, repetitions and precision (``baseline``: its value, e2e and clocks).  The reference itself cannot run.
* ``--impl reference``: the reference is TensorFlow-1.x example scripts; TF is not installable in this
  image (no wheel for Python 3.12, no network), so this arm reports ``unavailable`` (see DESIGN.md).
* ``--impl nccl``: the in-repo torch + NCCL + cuBLAS emulation of the same workflow (``baseline/``),
  for an apples-to-apples number on the same box.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl"])
    ap.add_argument("--mode", default="sync", choices=["sync", "async"])
    ap.add_argument("--optimizer", default="sgd", choices=["sgd", "momentum", "adam"])
    ap.add_argument("--lr", type=float, default=None, help="default: 0.001 for sgd/momentum (batch-SUM loss), 0.01 for adam")
    ap.add_argument("--hidden", type=int, default=100)
    ap.add_argument("--batch", type=int, default=100)
    ap.add_argument("--unroll", type=int, default=0, help="steps per CUDA graph (0: auto)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=-1, help="-1: min(steps, 1000); 0: skip")
    ap.add_argument("--e2e-prefetch", type=int, default=1, help="1: step t+1's H2D overlaps step t (double-buffered staging)")
    ap.add_argument("--graph-step", type=int, default=0,
                    help="resnet18: 1 = capture the worker's forward/backward into a CUDA graph after two eager steps")
    ap.add_argument("--ps-on-workers", type=int, default=1,
                    help="1 (default): N workers on N GPUs, ps shard s shares worker s's GPU and stream; 0 = --ps-only-task 1")
    ap.add_argument("--ps-only-task", type=int, default=0, help="1: ranks 0..num_ps-1 are ps-only tasks (1 ps + (N-1) workers)")
    ap.add_argument("--precision", default="tf32", choices=["tf32", "bf16"],
                    help="tf32: fp32 storage, TF32 MMAs, one-kernel worker step (reference precision); bf16: config 3")
    ap.add_argument("--step-ctas", type=int, default=0, help="tf32: CTAs of the step kernel (0: widest even split of the features)")
    ap.add_argument("--min-ms", type=float, default=100.0, help="e2e arms: collect at least this much timed region (repetitions of K steps)")
    ap.add_argument("--max-reps", type=int, default=400)
    ap.add_argument("--baseline", type=int, default=1, help="1: also time the torch+NCCL+cuBLAS arm in this invocation -> vs_baseline")
    ap.add_argument("--e2e-native-loop", type=int, default=1,
                    help="1: third e2e arm = PSTrainEngine.train_loop(x_batches_pinned, y_batches_pinned, steps): the same per-step "
                         "H2D copy / kernels / D2H loss read, K steps enqueued by one native call (csrc/step_exec.cu dtf_run_loop)")
    ap.add_argument("--e2e-native-timeout", type=float, default=120.0,
                    help="native-loop arm dead-man timer (s): if the arm has not returned by then, the record measured so far is "
                         "printed (native_loop_error = the timeout, no baseline arm) and the process ends")
    ap.add_argument("--e2e-depth", type=int, default=4, help="native loop: steps the host may run ahead of the landed losses")
    ap.add_argument("--e2e-pipeline", type=int, default=1,
                    help="1 (one-GPU runs and every-rank-a-worker topologies): also time step(..., sync_loss='deferred') -- the loss of step t is read after "
                         "step t+1 was enqueued -- and report the better arm, both kept under e2e.synchronous/.pipelined; "
                         "2: do so on every topology without the fallback to the synchronous number; 0: off")
    ap.add_argument("--publish", action="store_true", help="ps stores params into worker replicas (push-publish)")
    ap.add_argument("--num-train", type=int, default=55000)
    ap.add_argument("--f1-splits", type=int, default=1, help="split-K CTAs for the first GEMM")
    ap.add_argument("--head-ctas", type=int, default=8, help="row-parallel CTAs of the fused MLP head")
    ap.add_argument("--f1-block-n", type=int, default=64)
    ap.add_argument("--b3-block-n", type=int, default=64)
    ap.add_argument("--in-graph", action="store_true", help="ONE process drives all --gpus devices (in-graph replication)")
    ap.add_argument("--num-ps", type=int, default=0,
                    help="ps shards; 0 = auto: 1 for the MNIST MLP (0.3 MB of parameters: one apply kernel is the latency floor), "
                         "one per GPU for ResNet-18 with the shards on the workers' GPUs (45 MB: every GPU reduces / publishes 1/N)")
    ap.add_argument("--placement", default="greedy", choices=["round_robin", "greedy"],
                    help="ResNet-18 variables -> ps shards: replica_device_setter's round robin, or its GreedyLoadBalancingStrategy "
                         "by bytes (creation order, least-loaded shard)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed steps computed (last loss, parameters, optimizer slots) as DIR/<name>.npy")
    ap.add_argument("--model", default="mnist_mlp", choices=["mnist_mlp", "resnet18"],
                    help="resnet18: BASELINE.json config 5 (conv model under the same ps API; bandwidth-relevant: 44.7 MB per push)")
    ap.add_argument("--nvls", default="auto", choices=["off", "on", "auto"],
                    help="symmetric buffers + NVLS multicast: gradients reduced in the switch (multimem.ld_reduce), "
                         "parameters published with multimem.st")
    return ap.parse_args()


class ClockSampler:
    """SM clock / throttle-reason sampler running DURING the timed region (B200_PROFILING.md clocks line).

    In-process NVML polling (2 ms period) of THIS rank's GPU, so even a timed region of a few tens of milliseconds
    gets samples; falls back to an ``nvidia-smi -i <gpu> -lms`` subprocess when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 2):
        self.gpu, self.rows, self.proc = gpu_index, [], None
        self.period = period_ms
        self.nvml = None
        self._stop = False
        self.thread = None

    # -- NVML path ------------------------------------------------------------------------------------------------
    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        h = None
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            h = None
        if h is None:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(t.strip().isdigit() for t in vis.split(",")) and self.gpu < len(vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        return pynvml, h

    def _poll_nvml(self):
        pynvml, h = self.nvml
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop:
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                rs = int(get_reasons(h))
                try:
                    pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                self.rows.append((time.time(), float(sm), rs, pw))
            except Exception:
                pass
            time.sleep(self.period / 1000.0)

    def start(self):
        try:
            self.nvml = self._nvml_handle()
            pynvml, h = self.nvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.smi_period = 50
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.smi_period)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
            t_end = time.time() + 5.0
            while not self.rows and time.time() < t_end:     # the first nvidia-smi sample can take a second
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _read_smi(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        try:
            return self._stop_impl(t0, t1)
        except Exception as e:      # a sampling problem must never cost the measurement itself
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["sampler error: %r" % (e,)]}

    def _stop_impl(self, t0: float, t1: float):
        if self.nvml is not None:
            time.sleep(self.period / 1000.0 * 2)
            self._stop = True
            self.thread.join(timeout=1.0)
            inside = [r for r in self.rows if t0 <= r[0] <= t1]
            note = None
            if not inside:
                inside = sorted(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:2]
                note = "timed region shorter than the sampling period: nearest samples"
            if not inside:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "source": "nvml"}
            pynvml = self.nvml[0]
            bits = 0
            for r in inside:
                bits |= r[2]
            names = (("hw_slowdown", "HwSlowdown", 0x8), ("hw_thermal_slowdown", "HwThermalSlowdown", 0x40),
                     ("sw_thermal_slowdown", "SwThermalSlowdown", 0x20), ("sw_power_cap", "SwPowerCap", 0x4),
                     ("hw_power_brake_slowdown", "HwPowerBrakeSlowdown", 0x80))
            reasons = []
            for out_name, nv, default in names:
                mask = getattr(pynvml, "nvmlClocksEventReason" + nv, getattr(pynvml, "nvmlClocksThrottleReason" + nv, default))
                if bits & int(mask):
                    reasons.append(out_name)
            pws = [r[3] for r in inside if r[3] is not None]
            out = {"sm_mhz": statistics.median(r[1] for r in inside), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                   "samples": len(inside), "power_w_max": max(pws) if pws else None, "source": "nvml"}
            if note:
                out["note"] = note
            return out
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi and NVML unavailable"]}
        time.sleep(self.smi_period / 1000.0 * 1.5)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        mine = []
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8:
                mine.append((ts, f))
        inside = [f for ts, f in mine if t0 <= ts <= t1 + self.smi_period / 1000.0] or [f for _, f in mine[-3:]]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "source": "nvidia-smi"}
        sm = [float(f[1]) for f in inside]
        reasons = []
        for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6), ("sw_power_cap", 7)):
            if any(f[col].lower().startswith("active") for f in inside):
                reasons.append(name)
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(inside[0][2]), "reasons": reasons,
                "samples": len(inside), "source": "nvidia-smi", "power_w_max": max(float(f[3]) for f in inside if f[3].replace(".", "").isdigit())
                if any(f[3].replace(".", "").isdigit() for f in inside) else None}


def repetition_plan(K: int):
    """(repetitions, steps per repetition) of a timed region of exactly K steps: the most repetitions (<= 10) of equal length
    that keep each at >= 100 steps, so that a repetition is long against the launch of its first graph."""
    reps = max([r for r in range(1, 11) if K % r == 0 and K // r >= 100] or [1])
    return reps, K // reps


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays) -> None:
    """``arrays``: name -> array.  Written as ``out_dir/<name>.npy`` in float32 (float64 stays float64); when they exceed
    DUMP_BYTES in all, every array is cut to its share by a fixed, seeded sample of its elements (same positions every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {n: np.asarray(a, dtype=np.float64 if np.asarray(a).dtype == np.float64 else np.float32) for n, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, int(a.size * DUMP_BYTES // total))
            if keep < a.size:
                idx = np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))
                a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name.replace("/", "_") + ".npy"), a)


def reference_arm(args):
    why = ("reference is 7 TensorFlow-1.x scripts with no setup.py; tensorflow 1.x has no wheel for "
           "Python 3.12 and /opt/wheelhouse has none (pip install --no-index fails), so it cannot run here")
    print(json.dumps({"impl": "reference", "unavailable": why, "metric": "MNIST MLP samples/sec", "n_gpus": args.gpus}))


def greedy_shards(shapes, num_ps: int):
    """``tf.contrib.training.GreedyLoadBalancingStrategy(num_ps, byte_size_load_fn)`` under ``replica_device_setter``: variables in
    creation order, each to the ps task carrying the fewest bytes so far (ties: the lowest task)."""
    load, out = [0] * num_ps, []
    for _, shp in shapes:
        t = min(range(num_ps), key=load.__getitem__)
        n = 4
        for d in shp:
            n *= int(d)
        load[t] += n
        out.append(t)
    return out


def run_resnet18(args, rank, world, local_rank):
    """ResNet-18 (CIFAR stem, 11.2 M parameters) under the same fabric ps protocol: conv-as-tcgen05-GEMM workers,
    fused ps_apply (momentum), sync replicas.  Timed exactly like the headline: CUDA events, barrier + synchronize on
    both sides, max over ranks; every step copies its batch from pinned host memory and reads the loss back."""
    import torch
    import torch.distributed as dist
    from distributed_tensorflow_b200.models import resnet18_init, resnet18_loss, resnet18_param_shapes
    from distributed_tensorflow_b200.ops import cuda_lib
    from distributed_tensorflow_b200.parallel.fabric import Fabric
    from distributed_tensorflow_b200.parallel.generic_engine import GenericPSEngine
    from distributed_tensorflow_b200.parallel.ps_engine import EngineConfig
    N = args.gpus
    if N > 1 and world == 1:
        raise SystemExit("--model resnet18 with --gpus %d: launch one process per GPU with torch.distributed.run" % N)
    B = args.batch if args.batch != 100 else 64
    nvls = {"off": False, "on": True, "auto": "auto"}[args.nvls]
    opt = {"kind": "momentum", "lr": args.lr or 0.05, "momentum": 0.9}
    if N == 1:
        cfg = EngineConfig(num_ps=1, num_workers=1, colocated=True, optimizer=opt)
        fabric = Fabric(1, {0: local_rank})
    else:
        pow_ = bool(args.ps_on_workers)
        cfg = EngineConfig(num_ps=args.num_ps, num_workers=N if pow_ else N - args.num_ps, optimizer=opt, nvls=nvls,
                           ps_on_workers=pow_)
        fabric = Fabric.from_torch_distributed()
    shapes = resnet18_param_shapes(10, "cifar")
    shards = greedy_shards(shapes, cfg.num_ps) if (cfg.num_ps > 1 and args.placement == "greedy") else None
    eng = GenericPSEngine(shapes, cfg, fabric, shards=shards)
    eng.init_params(resnet18_init(10, "cifar", seed=2))
    nparams = sum(eng.shard_elems)
    is_worker = any(r in eng.worker_ranks for r in eng.ranks)
    my = next(iter(eng.ranks))
    rk = eng.ranks[my]
    nb = 64                                   # 64 pinned batches x B x 32x32x3 fp32 (50 MB at B=64), cycled
    g = torch.Generator().manual_seed(5 + rank)
    hx = torch.randn(nb, B, 32, 32, 3, generator=g).pin_memory() if is_worker else None
    hy = torch.eye(10)[torch.randint(0, 10, (nb, B), generator=g)].pin_memory() if is_worker else None

    def barrier():
        eng.synchronize()
        if world > 1:
            dist.barrier()
        eng.synchronize()

    losses = []

    def step(i):
        if is_worker:
            with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
                x = hx[i % nb].to(rk.device, non_blocking=True)
                y = hy[i % nb].to(rk.device, non_blocking=True)
            loss = eng.worker_step(my, resnet18_loss, x, y, graph=bool(args.graph_step))
            if my in eng.ps_ranks:
                eng.ps_apply(my)
            losses.append(float(loss))        # D2H read of the step's loss
        else:
            eng.ps_apply(my)
    K, W = args.steps if args.steps != 2000 else 20, max(3, min(args.warmup, 5))
    for i in range(W):
        step(i)
    barrier()
    eng.check_errors()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    barrier()
    n0 = cuda_lib.launch_count()
    t0 = time.time()
    with torch.cuda.device(rk.device):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(rk.stream)
    for i in range(K):
        step(W + i)
    e1.record(rk.stream)
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    ms_local = e0.elapsed_time(e1)
    stats = torch.tensor([ms_local, float(cuda_lib.launch_count() - n0)], dtype=torch.float64, device="cuda")
    if world > 1:
        mx, sm = stats.clone(), stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, launches = float(mx[0]), int(sm[1])
    else:
        ms, launches = ms_local, int(stats[1])
    eng.check_errors()
    value = cfg.num_workers * B * K / (ms / 1e3)
    lt = torch.tensor([losses[W] if len(losses) > W else -1e30, losses[-1] if losses else -1e30], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(lt, op=dist.ReduceOp.MAX)           # the ps ranks have no loss: take a worker's
    losses = [float(lt[0]), float(lt[1])]
    out = {"metric": "ResNet-18 samples/sec (whole box, device-timed, max over ranks), sync-replica PS", "value": value,
           "unit": "samples/sec", "n_gpus": N, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "impl": "ours",
           "data": "synthetic CIFAR-shaped 32x32x3 from pinned host memory (H2D every step), random-init weights",
           "config": {"model": "ResNet-18 (CIFAR stem), %d parameters" % nparams, "per_worker_batch": B,
                      "global_batch": cfg.num_workers * B, "optimizer": "momentum", "mode": "sync",
                      "parallelism": "ps1+worker1 colocated" if N == 1 else "ps%d+worker%d between-graph%s" % (
                          cfg.num_ps, cfg.num_workers, ", ps shards on the first workers' GPUs" if cfg.ps_on_workers else ""),
                      "fused_nn": bool(cuda_lib.FUSED_NN), "graph_step": bool(args.graph_step),
                      "grad_bytes_per_push": nparams * 4, "param_bytes_per_pull": nparams * 4,
                      "fabric": ("nvls: multimem.ld_reduce push / multimem.st pull" if getattr(eng, "nvls_multicast", False)
                                 else "symmetric buffers, unicast" if getattr(eng, "nvls", False) else "unicast peer stores / loads"),
                      "l2": "64 distinct batches cycled; activations + 45 MB of parameters + gradients exceed L2 per step"},
           "clocks": clocks, "gpu_launches": launches,
           "e2e": {"value": value, "unit": "samples/sec", "h2d_bytes_per_step": B * (32 * 32 * 3 + 10) * 4, "d2h_bytes_per_step": 4,
                   "note": "the timed loop itself copies every batch from pinned host memory and reads the loss back"},
           "first_loss": losses[0] if losses else None, "final_loss": losses[-1] if losses else None}
    eng.close()
    if getattr(args, "baseline", 0):
        # the divisor for config 5: cuDNN + autograd + NCCL arm, same invocation / batch / topology
        try:
            from baseline.nccl_resnet import run_nccl_resnet
            base = run_nccl_resnet(args, rank, world, local_rank, sampler_cls=ClockSampler)
            out["baseline"] = base
            out["vs_baseline"] = value / base["value"] if base.get("value") else None
        except Exception as e:          # noqa: BLE001
            if world > 1:
                raise
            out["baseline"] = {"error": repr(e)[:300]}
    return out


class CudaStreamTimer:
    """Device time of a region: CUDA events on every local rank's stream (max over them), read after a synchronize."""

    def start(self, eng):
        import torch
        evs = []
        for r, rk in eng.ranks.items():
            with torch.cuda.device(rk.device):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(rk.stream)
                evs.append((e0, e1, rk))
        return evs

    def stop(self, evs, eng) -> float:
        for e0, e1, rk in evs:
            e1.record(rk.stream)
        eng.synchronize()
        return max(e0.elapsed_time(e1) for e0, e1, _ in evs)


class DeadMan:
    """Dead-man timer around an arm that enqueues work from native code: if the arm neither returns nor raises within
    ``seconds`` (a hung stream / event wait cannot be cancelled from Python), ``on_fire()`` runs on the timer thread -- it
    prints the record measured so far -- and the process ends with status 0; the arms measured before it stand."""

    def __init__(self, seconds, on_fire, exit_fn=os._exit):
        self.fired = False
        self._t = None
        if on_fire is not None and seconds and seconds > 0:
            def fire():
                self.fired = True
                try:
                    on_fire()
                    sys.stdout.flush()
                finally:
                    exit_fn(0)
            self._t = threading.Timer(seconds, fire)
            self._t.daemon = True
            self._t.start()

    def cancel(self):
        if self._t is not None:
            self._t.cancel()


def run_e2e(eng, args, spec, K, num_workers, is_worker, world, pow_, images, labels, barrier, allmax, timer=None, pin=None,
            failsafe=None):
    """The end-to-end arms: the same metric through the public API with, every step, the H2D copy of that step's batch from
    pinned host memory and a D2H read of the step's loss -- ``step()`` synchronous, ``step(sync_loss="deferred")`` pipelined,
    ``train_loop()`` (K steps per native call); same repetition protocol as the device-timed number.  ``timer`` / ``pin`` are
    injected so that this logic also runs against a stand-in engine on CPU (tests/test_bench_e2e_logic.py)."""
    import torch
    timer = timer or CudaStreamTimer()
    pin = pin or (lambda a: torch.from_numpy(a).pin_memory())
    hx = hy = None
    if is_worker:
        n_use = min(args.num_train, 20000)
        hx = pin(images[:n_use])
        hy = pin(labels[:n_use])
        nb = n_use // spec.batch
    wl = [r for r in eng.ranks if r in eng.worker_ranks]
    woff = eng.worker_ranks.index(wl[0]) if wl else 0
    views = [(hx[b * spec.batch:(b + 1) * spec.batch], hy[b * spec.batch:(b + 1) * spec.batch]) for b in range(nb)] \
        if is_worker else []
    ctr = [0]
    last = [None]

    def batch_of(i):
        return views[(i * num_workers + woff) % nb]

    def e2e_k_steps():
        # every step: H2D of THIS step's batch from pinned host memory (issued one step ahead on the copy stream
        # = input double buffering, overlapping the previous step's kernels) + D2H read of this step's loss
        for _ in range(K):
            i = ctr[0]
            if is_worker:
                x, y = batch_of(i)
                last[0] = eng.step(x, y, sync_loss=True, prefetch=batch_of(i + 1) if args.e2e_prefetch else None)
            else:
                eng.step(sync_loss=False)
            ctr[0] += 1

    def e2e_k_steps_pipelined():
        # same copies every step, but step t+1 is enqueued BEFORE step t's loss is waited for (PendingLoss): the
        # host's turnaround overlaps the GPU's work on step t; every loss is still read back, one step late
        pending = None
        for _ in range(K):
            i = ctr[0]
            if not is_worker:
                eng.step(sync_loss=False)
            else:
                x, y = batch_of(i)
                h = eng.step(x, y, sync_loss="deferred", prefetch=batch_of(i + 1))
                if pending is not None:
                    last[0] = pending.result()
                pending = h
            ctr[0] += 1
        if pending is not None:
            last[0] = pending.result()

    hx3 = hx[:nb * spec.batch].view(nb, spec.batch, spec.in_dim) if is_worker else None
    hy3 = hy[:nb * spec.batch].view(nb, spec.batch, spec.classes) if is_worker else None

    def e2e_k_steps_native():
        # same per-step work (H2D of THIS step's batch one step ahead on the copy stream, the step's kernels, D2H of the
        # step's loss row), but the K steps are enqueued by ONE native call; the host reads every loss, at most
        # --e2e-depth steps late
        if is_worker:
            ls = eng.train_loop(hx3, hy3, K, first=(ctr[0] * num_workers + woff) % nb, stride=num_workers, depth=args.e2e_depth,
                                prefetch_next=bool(args.e2e_prefetch))
            last[0] = float(ls[-1])
            if not all(math.isfinite(float(v)) for v in ls):
                raise RuntimeError("native loop returned a non-finite loss")
        else:
            for _ in range(K):
                eng.step(sync_loss=False)
        ctr[0] += K

    def align_e2e():
        for _ in range(2):
            if is_worker:
                x, y = batch_of(ctr[0])
                # the loop is continuous across the untimed / timed boundary: the batch of the next step is already
                # travelling (every timed step still issues one H2D copy: the one of the step after it)
                eng.step(x, y, sync_loss=False, prefetch=batch_of(ctr[0] + 1) if args.e2e_prefetch else None)
            else:
                eng.step(sync_loss=False)
            ctr[0] += 1

    def measure_e2e(body):
        for _ in range(6):           # both staging parities + the CUDA-graphed plans are built by the first steps
            align_e2e()
        times, total = [], 0.0
        while len(times) < 3 or (total < args.min_ms and len(times) < args.max_reps):
            barrier()
            align_e2e()
            handle = timer.start(eng)
            w0 = time.time()
            body()
            eng.join_streams()
            dev_ms = timer.stop(handle, eng)             # records the end events, synchronizes, reads the device time
            wall = (time.time() - w0) * 1e3
            times.append(allmax([max(dev_ms, 0.0), wall]))
            total += times[-1][0]
        eng.check_errors()
        return times

    et = measure_e2e(e2e_k_steps)
    ems = statistics.median(t[0] for t in et)
    per_step = num_workers * spec.batch * K
    e2e = {"value": per_step / (ems / 1e3), "unit": "samples/sec", "steps": K, "reps": len(et),
           "ms_per_step": ems / K, "wall_ms_per_step": statistics.median(t[1] for t in et) / K,
           "h2d_bytes_per_step": spec.batch * (spec.in_dim + spec.classes) * 4,
           "d2h_bytes_per_step": 4 * eng.head_ctas,          # the loss partials of the step kernel's / head's CTAs
           "api": "PSTrainEngine.step(x_pinned, y_pinned, prefetch=next) -> loss" if args.e2e_prefetch
           else "PSTrainEngine.step(x_pinned, y_pinned) -> loss",
           "input_double_buffering": bool(args.e2e_prefetch), "loss_read": "synchronous, every step",
           "last_loss": allmax([last[0] if last[0] is not None else -1e30])[0]}
    if args.e2e_pipeline and ((world == 1 and is_worker) or args.e2e_pipeline == 2 or pow_):
        # second arm of the same API: loss handles read one step late
        try:
            pt = measure_e2e(e2e_k_steps_pipelined)
            pems = statistics.median(t[0] for t in pt)
            plast = allmax([last[0] if last[0] is not None else -1e30])[0]
            if not math.isfinite(plast):
                raise RuntimeError("pipelined loop returned loss %r" % (plast,))
            sync_part = {k: e2e[k] for k in ("value", "ms_per_step", "wall_ms_per_step", "last_loss")}
            pipe_part = {"value": per_step / (pems / 1e3), "ms_per_step": pems / K,
                         "wall_ms_per_step": statistics.median(t[1] for t in pt) / K, "last_loss": plast}
            e2e["synchronous"], e2e["pipelined"] = sync_part, pipe_part
            if pipe_part["value"] > e2e["value"]:
                e2e.update(pipe_part)
                e2e["api"] = "PSTrainEngine.step(x_pinned, y_pinned, sync_loss='deferred', prefetch=next) -> PendingLoss; .result()"
                e2e["loss_read"] = "every step's loss is copied D2H behind its kernels and read by the host one step late"
        except Exception as e:      # noqa: BLE001 - keep the synchronous measurement
            if world > 1:
                raise                # ranks must not diverge
            e2e["pipelined_error"] = repr(e)[:300]
    if args.e2e_native_loop and len(wl) <= 1 and ((world == 1 and is_worker) or pow_):
        # third arm: the framework's own training loop (one native call per K steps).  A failure on any rank drops the
        # arm on every rank (the flag is agreed on before anything is recorded); the other arms' numbers stand.
        nt, nerr = None, None
        so_far = json.loads(json.dumps(e2e))
        so_far["native_loop_error"] = ("dead-man timer: the native-loop arm did not return within %g s; record printed by the "
                                       "timer, baseline arm not run" % getattr(args, "e2e_native_timeout", 0.0))
        guard = DeadMan(getattr(args, "e2e_native_timeout", 0.0), (lambda: failsafe(so_far)) if failsafe else None)
        try:
            nt = measure_e2e(e2e_k_steps_native)
        except Exception as e:      # noqa: BLE001
            nerr = repr(e)[:300]
        try:                         # the agreement is a collective: a rank that hangs in the arm keeps the others here
            nlast = allmax([last[0] if (last[0] is not None and nerr is None) else -1e30])[0]
            failed = allmax([1.0 if (nerr is not None or not math.isfinite(nlast)) else 0.0])[0] > 0
        finally:
            guard.cancel()
        if failed:
            e2e["native_loop_error"] = nerr or "non-finite loss %r or a failure on another rank" % (nlast,)
        else:
            nems = statistics.median(t[0] for t in nt)
            if "synchronous" not in e2e:
                e2e["synchronous"] = {k: e2e[k] for k in ("value", "ms_per_step", "wall_ms_per_step", "last_loss")}
            nat_part = {"value": per_step / (nems / 1e3), "ms_per_step": nems / K,
                        "wall_ms_per_step": statistics.median(t[1] for t in nt) / K, "last_loss": nlast}
            e2e["native_loop"] = dict(nat_part, depth=args.e2e_depth)
            if nat_part["value"] > e2e["value"]:
                e2e.update(nat_part)
                e2e["reps"] = len(nt)
                e2e["api"] = "PSTrainEngine.train_loop(x_batches_pinned, y_batches_pinned, steps=K) -> losses[K]"
                e2e["loss_read"] = ("every step's loss is copied D2H behind its kernels into its own pinned row; the host waits "
                                    "for row i-%d before enqueuing step i and reads all K rows" % args.e2e_depth)
                e2e["input_double_buffering"] = True
    return e2e


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
        return 0
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if args.in_graph and world > 1:
        raise SystemExit("--in-graph runs as ONE process (do not launch it with torchrun)")
    if args.gpus > 1 and world == 1 and not args.in_graph:
        # `python bench.py --gpus N` without torchrun: one client process drives all N GPUs (in-graph replication)
        args.in_graph = True
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if args.impl == "nccl":
        from baseline.nccl_ps import run_nccl_baseline
        out = run_nccl_baseline(args, rank, world, local_rank)
        if rank == 0:
            print(json.dumps(out))
        if world > 1:
            dist.destroy_process_group()
        return 0

    from distributed_tensorflow_b200.ops import cuda_lib
    from distributed_tensorflow_b200.parallel.fabric import Fabric
    from distributed_tensorflow_b200.parallel.ps_engine import EngineConfig, MLPSpec, PSTrainEngine
    from distributed_tensorflow_b200.utils.mnist_data import synthetic_mnist

    if args.num_ps <= 0:
        args.num_ps = args.gpus if (args.model == "resnet18" and args.ps_on_workers and not args.ps_only_task) else 1
    if args.model == "resnet18":
        out = run_resnet18(args, rank, world, local_rank)
        if rank == 0:
            print(json.dumps(out))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    N = args.gpus
    spec = MLPSpec(hidden=args.hidden, batch=args.batch)
    if args.lr is None:
        args.lr = 0.01 if args.optimizer == "adam" else 0.001
        if args.mode == "async" and args.optimizer != "adam":
            args.lr /= max(1, args.gpus - (0 if (args.ps_on_workers and not args.ps_only_task) else args.num_ps))   # every push is applied alone
    opt = {"kind": args.optimizer, "lr": args.lr, "momentum": 0.9}
    pow_ = bool(args.ps_on_workers) and not bool(args.ps_only_task) and N > 1
    nw = N if pow_ else N - args.num_ps
    NVLS = {"off": False, "on": True, "auto": "auto"}[args.nvls]
    if args.in_graph and args.nvls == "auto":
        NVLS = False            # one-process topology: opt in with --nvls on
    common = dict(sync=args.mode == "sync", optimizer=opt, publish_replicas=args.publish, nvls=NVLS, f1_splits=args.f1_splits,
                  head_ctas=args.head_ctas, f1_block_n=args.f1_block_n, b3_block_n=args.b3_block_n, precision=args.precision, step_ctas=args.step_ctas)
    if args.in_graph and N > 1:
        cfg = EngineConfig(num_ps=args.num_ps, num_workers=nw, ps_on_workers=pow_, **common)
        fabric = Fabric(N, {r: r for r in range(N)})
    elif N == 1:
        cfg = EngineConfig(num_ps=1, num_workers=1, colocated=True, **common)
        fabric = Fabric(1, {0: local_rank})
    else:
        cfg = EngineConfig(num_ps=args.num_ps, num_workers=nw, ps_on_workers=pow_, **common)
        fabric = Fabric.from_torch_distributed()
    eng = PSTrainEngine(spec, cfg, fabric)
    eng.init_params()
    is_worker = any(r in eng.worker_ranks for r in eng.ranks)
    num_workers = cfg.num_workers

    # ---- data: synthetic MNIST-shaped train split (fp32, 172 MB) in every worker's HBM -----------------------
    images = labels = None
    if is_worker:
        images, labels = synthetic_mnist(args.num_train, seed=1)
        for r in eng.ranks:
            if r in eng.worker_ranks:
                eng.attach_dataset(r, images, labels)

    def barrier():
        eng.synchronize()
        if world > 1:
            dist.barrier()
        eng.synchronize()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    K, W = args.steps, max(args.warmup, 3)
    n_reps, k_rep = repetition_plan(K)
    use_graph = not args.no_graph
    unroll = args.unroll or next(u for u in (50, 40, 32, 25, 20, 16, 10, 8, 5, 4, 2, 1) if k_rep % u == 0)
    # ---- warm-up (eager: first-launch setup) + graph capture + graph warm-up ---------------------------------
    eng.enqueue_local_steps(W, "dataset")
    barrier()
    eng.check_errors()
    if use_graph:
        eng.capture_graphs(unroll, "dataset")
        k_graphs = eng._graphs
        eng.capture_graphs(2, "dataset")          # two untimed alignment steps in front of every timed repetition
        align_graphs = eng._graphs
        eng._graphs = k_graphs
        eng.replay_graphs(1)
        barrier()
        eng.check_errors()

    def align_steps():
        if use_graph:
            eng._graphs = align_graphs
            eng.replay_graphs(1)
            eng._graphs = k_graphs
        else:
            eng.enqueue_local_steps(2, "dataset")

    def k_steps():
        if use_graph:
            eng.replay_graphs(k_rep // unroll)
            if k_rep % unroll:
                eng.enqueue_local_steps(k_rep % unroll, "dataset")
        else:
            eng.enqueue_local_steps(k_rep, "dataset")

    def measure(body):
        """``n_reps`` repetitions of ``k_rep`` steps (K in all): barrier + synchronize, two untimed alignment steps (the sync
        protocol itself lines the ranks up, so the start skew of the barrier release is not part of the measurement), CUDA
        events on every local stream around the repetition's steps, MAX over ranks."""
        times = []
        for _ in range(n_reps):
            barrier()
            align_steps()
            evs = []
            for r, rk in eng.ranks.items():
                with torch.cuda.device(rk.device):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(rk.stream)
                    evs.append((e0, e1, rk))
            body()
            eng.join_streams()
            for e0, e1, rk in evs:
                e1.record(rk.stream)
            eng.synchronize()
            times.append(allmax([max(e0.elapsed_time(e1) for e0, e1, _ in evs)])[0])
        return times

    # ---- timed region ---------------------------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    barrier()
    launches0 = cuda_lib.launch_count()
    t0 = time.time()
    times = measure(k_steps)
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    reps = len(times)
    # kernels launched by the K timed steps only (the alignment steps are untimed and not counted)
    launched = cuda_lib.launch_count() - launches0
    per_align = 2 * sum((eng.launches_per_worker_step("dataset") if r in eng.worker_ranks else 0) +
                        ((1 if cfg.sync else num_workers) if r in eng.ps_ranks else 0) for r in eng.ranks)
    launches = launched - reps * per_align
    eng.check_errors()
    ms = statistics.median(times) * n_reps           # a K-step region at the median repetition's rate
    st = torch.tensor([float(launches)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(st, op=dist.ReduceOp.SUM)
    launches_total = int(st[0])
    value = num_workers * spec.batch * K / (ms / 1e3)
    loss = eng.read_loss() if is_worker else None
    loss = allmax([loss if loss is not None else -1e30])[0]
    gstep = eng.read_ctl(0, "global_step") if 0 in eng.ranks else None
    stale = eng.staleness() if (args.mode == "async" and 0 in eng.ranks) else None
    if args.dump_outputs and rank == 0:
        sd = eng.state_dict()
        dump_outputs(args.dump_outputs, dict({"loss": [loss]}, **{k: v.double().numpy() if k == "global_step" else v.float().numpy()
                                                                   for k, v in sd.items()}))

    # ---- ps traffic implied by the measured step time (BASELINE metric: push/pull GB/s vs 900 GB/s/dir) -----------
    # true-shape bytes: gradients travel as fp32, parameters as fp32 (tf32 engines) / bf16 replicas; every worker moves both every step.
    n_params = spec.in_dim * spec.hidden + spec.hidden + spec.hidden * spec.classes + spec.classes
    step_s = ms / K / 1e3
    push_b, pull_b = 4 * n_params, (4 if args.precision == "tf32" else 2) * n_params
    traffic = {"params": n_params, "push_bytes_per_worker_step": push_b, "pull_bytes_per_worker_step": pull_b,
               "ps_ingest_gbps": num_workers * push_b / step_s / 1e9 / max(1, cfg.num_ps),
               "ps_egress_gbps": num_workers * pull_b / step_s / 1e9 / max(1, cfg.num_ps),
               "note": "effective rate per ps shard over the whole step (latency-bound at this model size: 0.3 MB per push); "
                       "link-rate measurements of the same kernels at large payloads: profiles/nvls_check_*.json"}
    traffic["ps_ingest_fraction_of_900"] = traffic["ps_ingest_gbps"] / 900.0
    traffic["ps_egress_fraction_of_900"] = traffic["ps_egress_gbps"] / 900.0
    nvls_on, mc_on = bool(getattr(eng, "nvls", False)), bool(getattr(eng, "nvls_multicast", False))

    def build_out(e2e, base):
        out = {
            "metric": "MNIST MLP samples/sec (whole box, device-timed, max over ranks), sync-replica PS",
            "value": value, "unit": "samples/sec", "n_gpus": N, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (value / base["value"]) if base and base.get("value") else None,
            "dtype": args.precision,
            "data": "synthetic MNIST-shaped 28x28 (55000x784 fp32 in HBM), random-init weights",
            "impl": "ours", "reps": reps, "timed_ms_total": sum(times),
            "ms_per_step_min_max": [min(times) / k_rep, max(times) / k_rep],
            "config": {"model": "MNIST MLP 784-%d-10, clipped batch-sum xent" % spec.hidden,
                       "global_batch": num_workers * spec.batch, "per_worker_batch": spec.batch,
                       "parallelism": ("ps1+worker1 colocated on one GPU" if N == 1 else "ps%d+worker%d %s%s" % (
                           cfg.num_ps, cfg.num_workers, "in-graph (one client process)" if args.in_graph else "between-graph",
                           ", ps shards on the first workers' GPUs" if cfg.ps_on_workers else "")),
                       "mode": args.mode, "optimizer": args.optimizer, "lr": args.lr,
                       "precision": ("fp32 storage, TF32 tensor-core multiply, fp32 accumulate" if args.precision == "tf32"
                                     else "bf16 operands, fp32 accumulate"),
                       "worker_step": ("one kernel (csrc/mlp_step.cu)" if args.precision == "tf32" else "stage + GEMM + head + GEMM"),
                       "l2": "inputs larger than L2: 172 MB fp32 train split cycled in HBM",
                       "timing": "median of %d repetitions of exactly %d steps (%d timed steps), each after barrier + 2 untimed "
                                 "alignment steps" % (reps, k_rep, K),
                       "cuda_graph_unroll": unroll if use_graph else 0,
                       "pull": ("nvls multimem.st publish into fp32/bf16 replicas" if nvls_on and mc_on
                                else "publish-replicas" if (args.publish or nvls_on) else "peer-pull by TMA inside the step / GEMM kernel"),
                       "push": ("local store + nvls multimem.ld_reduce on the ps" if nvls_on and mc_on else
                                "local store + ps peer loads" if nvls_on else "peer stores from the TMEM epilogue")},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_total, "ps_traffic": traffic,
            "final_loss": loss, "global_step": gstep, "staleness": stale,
        }
        if base is not None:
            out["baseline"] = {k: base.get(k) for k in ("impl", "value", "ms_per_step", "reps", "clocks", "e2e", "error", "config")
                               if base.get(k) is not None}
            if e2e and base.get("e2e") and base["e2e"].get("value"):
                out["vs_baseline_e2e"] = e2e["value"] / base["e2e"]["value"]
        return out

    def failsafe(e2e_so_far):
        # runs on the dead-man timer's thread when the native-loop arm hangs: the numbers measured so far are the record
        if rank == 0:
            print(json.dumps(build_out(e2e_so_far, None)))

    # ---- end-to-end: public API step(x, y) with H2D of the batch and D2H of the loss every step -----------------
    e2e = None
    if args.e2e_steps != 0:
        e2e = run_e2e(eng, args, spec, K, num_workers, is_worker, world, pow_, images, labels, barrier, allmax, failsafe=failsafe)

    eng.close()

    # ---- the divisor: torch + NCCL + cuBLAS (CUDA-graphed) arm, same invocation / steps / repetitions / precision --------
    base = None
    if args.baseline and not args.in_graph:
        try:
            from baseline.nccl_ps import run_nccl_baseline
            bargs = argparse.Namespace(**vars(args))
            bargs.ps_on_workers, bargs.ps_only_task = int(pow_ or N == 1), int(not pow_ and N > 1)
            base = run_nccl_baseline(bargs, rank, world, local_rank, sampler_cls=ClockSampler, images=images, labels=labels)
        except Exception as e:          # noqa: BLE001 - the measured arm must survive a baseline problem
            if world > 1:
                raise
            base = {"error": repr(e)[:300]}

    if rank == 0:
        print(json.dumps(build_out(e2e, base)))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
