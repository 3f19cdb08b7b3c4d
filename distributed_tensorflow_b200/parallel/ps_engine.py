"""Fabric parameter-server engine: the B200 fast path for ps/worker training (SURVEY §7.3, §7.2 step 6/7).

Same semantics as the control-plane path (``train/sync_replicas.py`` + ``parallel/server.py``) --
variables placed on ps shards round-robin, workers pull parameters / push gradients, the ps applies
SGD/Momentum/TF-Adam, sync mode aggregates the MEAN of fresh gradients and hands out tokens, async
mode applies every push immediately and measures staleness -- but all of it runs on the GPUs:

* parameters, optimizer slots, per-worker gradient slots and the control block live in the ps GPU's
  HBM (padded flat layout); workers address them over NVLink peer memory (``parallel/fabric.py``);
* a worker step is three kernels of ours: ``gemm_bf16_tcgen05`` (x.W1 + b1, ReLU; its TMA producer
  first acquires the token and then loads W1 tiles straight from the ps -- *pull fused into the
  first GEMM*), ``mlp_head`` (logits, softmax, clipped xent, dlogits, dW2/db2/db1 pushed to the ps,
  dh), ``gemm_bf16_tcgen05`` (dW1 = x^T.dh whose epilogue stores the tiles into the ps gradient
  slot and release-increments the arrival counter -- *push fused into the backward GEMM*);
* the ps step is one kernel: ``ps_apply`` (wait for arrivals -> N-way reduce -> mean -> apply ->
  publish bf16 shadow -> release tokens).

``EngineConfig.precision`` selects the worker's arithmetic: ``"tf32"`` (default; the reference model is fp32,
/root/reference/distributed_mnist.py:98-113): parameters, activations and gradients stay fp32 in memory, the two large
GEMMs run as TF32 on the tensor cores, and the WHOLE worker step is ONE kernel (``csrc/mlp_step.cu``: token wait, W1
pulled by TMA as the B operand, fused head, dW1 pushed from TMEM, arrival) -- a step is two launches, worker + ps;
``"bf16"`` (BASELINE config 3): bf16 parameter replica and activations, the three-kernel chain described above.

No NCCL, cuBLAS or host round trip is on the step path.  ``torch.distributed`` is used once, to
exchange IPC handles, and by the benchmark for barriers.

Topologies: ``between-graph`` = one process per GPU (``Fabric.from_torch_distributed``); ``in-graph``
= one process drives every GPU (all ranks local).  Ranks ``0..num_ps-1`` are ps shards, the rest are
workers; with a single GPU the ps and the worker share it (and its stream).
"""
from __future__ import annotations

import contextlib
import ctypes
import math
import os
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from ..ops import cuda_lib
from ..ops.cuda_lib import MAX_WORKERS, GemmArgs, MlpHeadArgs, MlpStepArgs, PsApplyArgs, round_up
from .fabric import Fabric, FabricBuffer, view_tensor

__all__ = ["MLPSpec", "EngineConfig", "PSTrainEngine", "PendingLoss", "smoke_step", "VarLayout"]


class PendingLoss:
    """The loss of a step whose device->host copy may still be in flight (``step(..., sync_loss="deferred")``).

    ``result()`` waits for THAT step's copy only (an event recorded right behind it on the compute stream) and
    returns the batch-sum loss; the host is free to enqueue the next step first, so the GPU never idles while
    Python comes back around the loop.  The equivalent in the reference's world is fetching ``loss`` one ``run``
    late; every step's loss is still read back (4 * head_ctas bytes) exactly once."""
    __slots__ = ("_event", "_host", "_n", "_value")

    def __init__(self, event, host, n: int, value: Optional[float] = None):
        self._event, self._host, self._n, self._value = event, host, int(n), value

    def done(self) -> bool:
        return self._value is not None or bool(self._event.query())

    def result(self) -> float:
        if self._value is None:
            self._event.synchronize()
            self._value = float(self._host[:self._n].sum())
            self._event = self._host = None
        return self._value

    __float__ = result

    def __repr__(self) -> str:
        return "PendingLoss(%s)" % ("%g" % self._value if self._value is not None else "in flight")


@dataclass
class MLPSpec:
    in_dim: int = 784
    hidden: int = 100
    classes: int = 10
    batch: int = 100


@dataclass
class EngineConfig:
    num_ps: int = 1
    num_workers: int = 1
    sync: bool = True
    replicas_to_aggregate: Optional[int] = None
    optimizer: Dict[str, Any] = field(default_factory=lambda: {"kind": "sgd", "lr": 0.01})
    clip_min: float = 1e-10
    publish_replicas: bool = False        # True: ps stores new params into every worker's replica (push-publish)
    colocated: bool = False               # single GPU: ps shard 0 and worker 0 share device + stream
    ps_on_workers: bool = False           # N GPUs, N workers: ps shard s lives on worker s's GPU and shares its stream (no GPU is
                                          # spent on a ps-only task; world == num_workers).  First hardware run pending.
    nvls: Any = False                     # True/"auto": symmetric VMM buffers -- gradients stay in the WORKERS' HBM and the
                                          # ps sums them with multimem.ld_reduce (in-switch), parameters are published with
                                          # ONE multimem.st stream into every GPU's replica ("auto": only if the box has NVLS)
    shards: Optional[Dict[str, int]] = None   # explicit ps shard of hid_w / hid_b / sm_w / sm_b (graph programs: from the variables'
                                          # device strings); default = round-robin in the reference's creation order
    step_ctas: int = 0                    # tf32: CTAs (= input-feature slices) of the step kernel; 0 = widest even split (784 -> 7 x 112)
    precision: str = "tf32"               # "tf32": fp32 storage, TF32 tensor-core GEMMs, one-kernel worker step (mlp_step.cu);
                                          # "bf16": bf16 replica / activations, GEMM + head + GEMM kernels
    f1_splits: int = 1                    # split-K CTAs for the first GEMM (fp32 atomic partials, bias+ReLU in the head)
    head_ctas: int = 8                    # row-parallel CTAs of the fused head (batch reductions via fp32 atomics)
    f1_block_n: int = 64                  # N tile of the forward GEMM (0: one tile covering `hidden`)
    b3_block_n: int = 64                  # N tile of the dW1 GEMM (0: one tile covering `hidden`)
    timeout_ns: int = 5_000_000_000
    loss_hist: int = 4096
    trace_cap: int = 4096
    worker_trace_cap: int = 1024     # rows of the per-worker step ring (mlp_step_kernel stamps one 64-byte row per launch)
    seed: int = 0


@dataclass
class VarLayout:
    name: str
    shape: Tuple[int, ...]
    shard: int
    offset: int          # element offset inside the shard's flat buffers
    rows: int
    cols: int
    pitch: int           # row pitch in elements (multiple of 8 -> 16-byte bf16 rows for TMA)

    @property
    def numel_padded(self) -> int:
        return self.rows * self.pitch


_KIND = {"sgd": 0, "momentum": 1, "adam": 2}


def _layout(spec: MLPSpec, num_ps: int, wide_pitch: bool = False, shards: Optional[Dict[str, int]] = None
            ) -> Tuple[Dict[str, VarLayout], List[int]]:
    """Round-robin placement in creation order (global_step, hid_w, hid_b, sm_w, sm_b), SURVEY A5.
    ``wide_pitch`` (fp32 / tf32 engines): rows of the large matrix are padded to whole 128-byte chunks (32 floats), so every
    row of a TMA box is one aligned line; the padding is zero and stays zero (its gradient is never written)."""
    order = [("global_step", ()), ("hid_w", (spec.in_dim, spec.hidden)), ("hid_b", (spec.hidden,)),
             ("sm_w", (spec.hidden, spec.classes)), ("sm_b", (spec.classes,))]
    sizes = [0] * num_ps
    out: Dict[str, VarLayout] = {}
    for i, (name, shape) in enumerate(order):
        shard = (shards[name] if shards and name in shards else i) % num_ps
        if name == "global_step":
            continue                      # lives in the shard-0 control block (K7)
        rows, cols = (shape[0], shape[1]) if len(shape) == 2 else (1, shape[0])
        pitch = round_up(cols, 32) if (wide_pitch and len(shape) == 2 and cols > 16) else round_up(cols, 8)
        off = round_up(sizes[shard], 64)
        out[name] = VarLayout(name, tuple(shape), shard, off, rows, cols, pitch)
        sizes[shard] = off + rows * pitch
    return out, [round_up(max(s, 64), 64) for s in sizes]


class _Rank:
    """Per-rank device state (buffers, stream, cached launch descriptors)."""

    def sync(self) -> None:
        self.stream.synchronize()
        if self.ps_stream is not None:
            self.ps_stream.synchronize()

    def __init__(self, rank: int, device: int):
        self.rank, self.device = rank, torch.device("cuda", device)
        self.stream: Optional[torch.cuda.Stream] = None
        self.ps_stream: Optional[torch.cuda.Stream] = None     # ps shard hosted next to a worker on another GPU's fabric: own stream
        self.step = 0                    # steps enqueued so far (worker) / applies enqueued (ps)
        self.bufs: Dict[str, FabricBuffer] = {}


class PSTrainEngine:
    def __init__(self, spec: MLPSpec, cfg: EngineConfig, fabric: Fabric):
        self.spec, self.cfg, self.fabric = spec, cfg, fabric
        self.lib = cuda_lib.load()
        if cfg.num_workers > MAX_WORKERS:
            raise ValueError("at most %d workers" % MAX_WORKERS)
        if spec.batch > 128 or spec.hidden > 256 or spec.classes > 16:
            raise ValueError("the fused MLP head handles batch<=128, hidden<=256, classes<=16")
        if cfg.precision not in ("tf32", "bf16"):
            raise ValueError("precision must be 'tf32' or 'bf16'")
        self.tf32 = cfg.precision == "tf32"
        if self.tf32 and (spec.hidden > 128 or cfg.num_ps > 4):
            raise ValueError("the one-kernel tf32 step handles hidden<=128 and <=4 ps shards; use precision='bf16'")
        self.world = fabric.world_size
        if cfg.colocated:
            assert self.world == 1 and cfg.num_ps == 1 and cfg.num_workers == 1
            self.ps_ranks, self.worker_ranks = [0], [0]
        elif cfg.ps_on_workers:
            # every rank is a worker; ranks 0..num_ps-1 additionally host a ps shard.  On such a rank the stream runs
            # [worker step t][ps_apply t][worker step t+1]...: the apply waits for the OTHER workers' arrivals while this
            # GPU's own step-t work is already done, and the next step needs the apply's token anyway, so sharing the
            # stream adds nothing to the critical path.
            assert self.world == cfg.num_workers and 1 <= cfg.num_ps <= self.world, "ps_on_workers: world = num_workers >= num_ps"
            self.ps_ranks = list(range(cfg.num_ps))
            self.worker_ranks = list(range(self.world))
        else:
            assert self.world == cfg.num_ps + cfg.num_workers, "world = num_ps + num_workers"
            self.ps_ranks = list(range(cfg.num_ps))
            self.worker_ranks = list(range(cfg.num_ps, self.world))
        self.layout, self.shard_elems = _layout(spec, cfg.num_ps, wide_pitch=self.tf32, shards=cfg.shards)
        self.R = cfg.replicas_to_aggregate or cfg.num_workers
        self.opt = dict(cfg.optimizer)
        self.kind = _KIND[self.opt["kind"]]
        self.ctl_bytes = self.lib.dtf_sizeof_ps_control()
        self.mb_bytes = self.lib.dtf_sizeof_mailbox()
        self.off = {k: self.lib.dtf_offsetof_ctl(i) for i, k in enumerate(
            ["global_step", "param_version", "beta1_power", "beta2_power", "dropped_stale", "applied_total",
             "staleness_hist", "staleness_sum", "err", "w", "w_stride", "consumed"])}
        self.ranks: Dict[int, _Rank] = {r: _Rank(r, d) for r, d in fabric.local_ranks.items()}
        for rk in self.ranks.values():
            with torch.cuda.device(rk.device):
                rk.stream = torch.cuda.Stream(rk.device)
                if cfg.ps_on_workers and rk.rank in self.ps_ranks and os.environ.get("DTF_PS_STREAM", "1") == "1":
                    # The shard's apply kernels run NEXT TO this GPU's worker kernels, not between them: everything they
                    # exchange goes through the same system-scope flags as with a remote worker, so no stream order is
                    # needed -- and the worker's next step (setup, batch prefetch, token wait) no longer queues behind
                    # the apply's launch + completion.
                    rk.ps_stream = torch.cuda.Stream(rk.device)
        # arrivals a complete push adds on each shard: 1 for the head (if it pushes there) + dW1 tiles
        lw = self.layout
        self.m_tiles_w1 = (spec.in_dim + 127) // 128
        self.ctas_per_push = [0] * cfg.num_ps
        head_shards = {lw["sm_w"].shard, lw["sm_b"].shard, lw["hid_b"].shard} - {lw["hid_w"].shard}
        self.head_ctas = max(1, min(int(cfg.head_ctas), 16))
        rows = (spec.batch + self.head_ctas - 1) // self.head_ctas
        rows = (rows + 7) // 8 * 8
        self.head_ctas = (spec.batch + rows - 1) // rows                 # what the launcher will actually use
        for s in head_shards:
            self.ctas_per_push[s] += self.head_ctas
        bn = 64 if spec.hidden <= 64 else (128 if spec.hidden <= 128 else (192 if spec.hidden <= 192 else 256))
        self.block_n_w1 = bn
        self.block_n_f1 = cfg.f1_block_n or bn
        self.block_n_b3 = cfg.b3_block_n or bn
        self.ctas_per_push[lw["hid_w"].shard] += self.m_tiles_w1 * ((spec.hidden + self.block_n_b3 - 1) // self.block_n_b3)
        if self.tf32:
            # one kernel of G CTAs does the whole step; every CTA signals every shard that holds one of the four variables
            ds = ctypes.c_int(0)
            self.step_ctas = int(self.lib.dtf_mlp_step_slices(spec.in_dim, spec.batch, ctypes.byref(ds)))
            self.step_slice = int(ds.value)
            if cfg.step_ctas:
                self.step_ctas = int(cfg.step_ctas)
                self.step_slice = round_up((spec.in_dim + self.step_ctas - 1) // self.step_ctas, 8)
                assert self.step_ctas <= 16 and self.step_slice <= 128 and (spec.batch + self.step_ctas - 1) // self.step_ctas <= 16
            self.head_ctas = self.step_ctas                        # loss partials per step
            self.var_shards = sorted({lw[v].shard for v in ("hid_w", "hid_b", "sm_w", "sm_b")})
            self.ctas_per_push = [self.step_ctas if s in self.var_shards else 0 for s in range(cfg.num_ps)]
        self._allocate()
        self._exchange()
        self._build_launches()

    # ------------------------------------------------------------------------------------------------
    # memory
    # ------------------------------------------------------------------------------------------------
    def _allocate(self) -> None:
        f, cfg, spec = self.fabric, self.cfg, self.spec
        W = cfg.num_workers
        # ---- NVLS mode: one symmetric gradient buffer and one symmetric bf16 replica per shard (collective allocs) ----
        want = cfg.nvls
        self.nvls, self.nvls_multicast = False, False
        self.sym_grads: List[Any] = []
        self.sym_repl: List[Any] = []
        if want and self.world > 1:
            level = f.nvls_level()
            if want == "auto" and level < 2:
                want = False
            elif level == 0:
                raise RuntimeError("nvls=True needs CUDA VMM (POSIX fd export); not available on this machine")
            elif self.tf32 and level < 2:
                want = False            # fp32 replicas are published with multimem.st only: no multicast -> unicast fabric
        if want and self.world > 1:
            self.nvls = True
            for s in range(cfg.num_ps):
                self.sym_grads.append(f.alloc_symmetric("sgrads%d" % s, self.shard_elems[s] * 4))
                # (+ 256 bytes behind the replica: the multicast token counter of the tf32 path, bumped by multimem.red)
                self.sym_repl.append(f.alloc_symmetric("srepl%d" % s, self.shard_elems[s] * (4 if self.tf32 else 2) + 256))
            self.nvls_multicast = self.sym_grads[0].multicast
        for r, rk in self.ranks.items():
            if r in self.ps_ranks:
                s = self.ps_ranks.index(r)
                n = self.shard_elems[s]
                for name, nbytes in (("ctl%d" % s, self.ctl_bytes), ("master%d" % s, n * 4), ("shadow%d" % s, n * 2),
                                     ("grads%d" % s, n * 4 * W), ("slot_m%d" % s, n * 4), ("slot_v%d" % s, n * 4),
                                     ("trace%d" % s, cfg.trace_cap * 32)):
                    if self.nvls and name.startswith("shadow"):
                        rk.bufs[name] = self.sym_repl[s].local(r)           # the ps's own copy of the replica
                    elif self.nvls and name.startswith("grads"):
                        rk.bufs[name] = self.sym_grads[s].local(r)          # stays zero: the ps contributes nothing
                    else:
                        rk.bufs[name] = f.alloc(r, name, nbytes)
                for name in ("ctl%d" % s, "master%d" % s) + (() if self.nvls else ("shadow%d" % s, "grads%d" % s)):
                    f.publish(r, name)
            if r in self.worker_ranks:
                w = self.worker_ranks.index(r)
                ldh = round_up(spec.hidden, 8)
                names = [("mailbox_w%d" % w, self.mb_bytes * cfg.num_ps),
                         ("x16_w%d" % w, 128 * spec.in_dim * 2), ("labels_w%d" % w, 128 * 16 * 4),
                         ("xf32_w%d" % w, 128 * spec.in_dim * 4),
                         ("h_w%d" % w, 128 * ldh * 2), ("dh_w%d" % w, 128 * ldh * 2), ("hacc_w%d" % w, 128 * ldh * 4),
                         ("misc_w%d" % w, 4096 + cfg.loss_hist * 4)]
                if self.tf32:
                    # scratch of the one-kernel step: partial pre-activations + dh + partial head gradients (L2 resident),
                    # 8 sync counters, phase stamps
                    nfl = (self.step_ctas * 128 * (round_up(spec.hidden, 16) + 4) + 128 * 128 + 64
                           + self.step_ctas * int(self.lib.dtf_mlp_step_head_part_floats()))
                    names += [("stepscr_w%d" % w, nfl * 4), ("stepflags_w%d" % w, 256), ("steptrace_w%d" % w, 16 * 32 * 8),
                              ("stepring_w%d" % w, (cfg.worker_trace_cap + 1) * 64)]
                for s in range(cfg.num_ps):
                    if self.nvls:
                        rk.bufs["replica%d_w%d" % (s, w)] = self.sym_repl[s].local(r)
                    else:
                        names.append(("replica%d_w%d" % (s, w), self.shard_elems[s] * 2))
                for name, nbytes in names:
                    rk.bufs[name] = f.alloc(r, name, nbytes)
                f.publish(r, "mailbox_w%d" % w)
                if cfg.publish_replicas and not self.nvls:
                    for s in range(cfg.num_ps):
                        f.publish(r, "replica%d_w%d" % (s, w))

    def _exchange(self) -> None:
        f, cfg = self.fabric, self.cfg
        self.peer: Dict[Tuple[int, str], FabricBuffer] = {}
        for r in self.ranks:
            if r in self.worker_ranks:
                for s, pr in enumerate(self.ps_ranks):
                    for base in ("ctl", "master") + (() if self.nvls else ("shadow", "grads")):
                        self.peer[(r, "%s%d" % (base, s))] = f.peer(r, pr, "%s%d" % (base, s))
            if r in self.ps_ranks:
                s = self.ps_ranks.index(r)
                for w, wr in enumerate(self.worker_ranks):
                    self.peer[(r, "mailbox_w%d" % w)] = f.peer(r, wr, "mailbox_w%d" % w)
                    if self.nvls:
                        # unicast views of every worker's copies: async / backup-worker reads, replica stores without NVLS
                        self.peer[(r, "sgrads%d_w%d" % (s, w))] = self.sym_grads[s].peer(r, wr)
                        self.peer[(r, "replica%d_w%d" % (s, w))] = self.sym_repl[s].peer(r, wr)
                    elif cfg.publish_replicas:
                        self.peer[(r, "replica%d_w%d" % (s, w))] = f.peer(r, wr, "replica%d_w%d" % (s, w))

    # ------------------------------------------------------------------------------------------------
    # parameter init / access (ps side)
    # ------------------------------------------------------------------------------------------------
    def _var_view(self, rk: _Rank, base: str, lay: VarLayout, dtype=torch.float32) -> torch.Tensor:
        buf = rk.bufs["%s%d" % (base, lay.shard)]
        es = 4 if dtype == torch.float32 else 2
        t = buf.tensor(dtype, lay.offset * es, lay.numel_padded)
        return t.view(lay.rows, lay.pitch)[:, :lay.cols]

    def init_params(self, values: Optional[Dict[str, torch.Tensor]] = None) -> None:
        """Chief-style initialisation on the ps shards (truncated normal / zeros like the reference model),
        then publish the bf16 shadow (+replicas) and the initial tokens."""
        spec, cfg = self.spec, self.cfg
        g = torch.Generator(device="cpu")
        g.manual_seed(cfg.seed)
        init = {}
        t = torch.empty(spec.in_dim, spec.hidden)
        torch.nn.init.trunc_normal_(t, 0.0, 1.0 / math.sqrt(spec.in_dim), -2.0 / math.sqrt(spec.in_dim),
                                    2.0 / math.sqrt(spec.in_dim), generator=g)
        init["hid_w"] = t
        init["hid_b"] = torch.zeros(spec.hidden)
        t2 = torch.empty(spec.hidden, spec.classes)
        sd = 1.0 / math.sqrt(spec.hidden)
        torch.nn.init.trunc_normal_(t2, 0.0, sd, -2 * sd, 2 * sd, generator=g)
        init["sm_w"] = t2
        init["sm_b"] = torch.zeros(spec.classes)
        if values:
            for k, v in values.items():
                init[k] = torch.as_tensor(v).float().reshape(self.layout[k].shape)
        for r, rk in self.ranks.items():
            if r not in self.ps_ranks:
                continue
            s = self.ps_ranks.index(r)
            with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
                for base in ("master", "slot_m", "slot_v", "grads", "shadow", "ctl"):
                    rk.bufs["%s%d" % (base, s)].tensor(torch.uint8).zero_()
                for name, lay in self.layout.items():
                    if lay.shard != s:
                        continue
                    v = init[name].reshape(lay.rows, lay.cols).to(rk.device)
                    self._var_view(rk, "master", lay).copy_(v)
                ctl = rk.bufs["ctl%d" % s]
                b = ctl.tensor(torch.float32, self.off["beta1_power"], 2)
                b[0] = float(self.opt.get("beta1", 0.9))
                b[1] = float(self.opt.get("beta2", 0.999))
                n = self.shard_elems[s]
                if self.tf32:
                    # fp32 end to end: workers read the master itself (same GPU / NVLink peer loads by TMA) or, under
                    # NVLS, their fp32 replica of it
                    if self.nvls:
                        m = rk.bufs["master%d" % s].tensor(torch.float32, 0, n)
                        rk.bufs["shadow%d" % s].tensor(torch.float32, 0, n).copy_(m)
                        for w in range(cfg.num_workers):
                            self.peer[(r, "replica%d_w%d" % (s, w))].tensor(torch.float32, 0, n).copy_(m)
                else:
                    rc = self.lib.dtf_ps_publish(rk.bufs["master%d" % s].ptr, rk.bufs["shadow%d" % s].ptr, n,
                                                 rk.stream.cuda_stream)
                    assert rc == 0, rc
                    if cfg.publish_replicas or self.nvls:
                        sh = rk.bufs["shadow%d" % s].tensor(torch.bfloat16, 0, n)
                        for w in range(cfg.num_workers):
                            self.peer[(r, "replica%d_w%d" % (s, w))].tensor(torch.bfloat16, 0, n).copy_(sh)
            rk.stream.synchronize()
        for r, rk in self.ranks.items():
            if r in self.worker_ranks:
                w = self.worker_ranks.index(r)
                with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
                    for name in ("mailbox_w%d" % w, "misc_w%d" % w, "x16_w%d" % w, "h_w%d" % w, "dh_w%d" % w,
                                 "labels_w%d" % w, "hacc_w%d" % w, "xf32_w%d" % w) + \
                            (("stepscr_w%d" % w, "stepflags_w%d" % w, "steptrace_w%d" % w, "stepring_w%d" % w) if self.tf32 else ()):
                        rk.bufs[name].tensor(torch.uint8).zero_()
                    for sg in self.sym_grads:
                        sg.local(r).tensor(torch.uint8).zero_()
                    for s_, sr in enumerate(self.sym_repl):       # the token counter behind the replica (multimem.red target)
                        sr.local(r).tensor(torch.uint8, self.shard_elems[s_] * (4 if self.tf32 else 2), 256).zero_()
                rk.stream.synchronize()
            rk.step = 0
        self.fabric.barrier()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """True-shape fp32 parameters + global_step gathered from the LOCAL ps shards (checkpointing)."""
        out: Dict[str, torch.Tensor] = {}
        for r, rk in self.ranks.items():
            if r not in self.ps_ranks:
                continue
            s = self.ps_ranks.index(r)
            rk.sync()
            for name, lay in self.layout.items():
                if lay.shard == s:
                    out[name] = self._var_view(rk, "master", lay).reshape(lay.shape).detach().cpu().clone()
                    if self.kind >= 1:
                        out[name + "/" + ("Momentum" if self.kind == 1 else "Adam")] = \
                            self._var_view(rk, "slot_m", lay).reshape(lay.shape).detach().cpu().clone()
                    if self.kind == 2:
                        out[name + "/Adam_1"] = self._var_view(rk, "slot_v", lay).reshape(lay.shape).detach().cpu().clone()
            if s == 0:
                out["global_step"] = torch.tensor(self.read_ctl(0, "global_step"), dtype=torch.int64)
                if self.kind == 2:
                    b = rk.bufs["ctl0"].tensor(torch.float32, self.off["beta1_power"], 2).cpu()
                    out["beta1_power"], out["beta2_power"] = b[0].clone(), b[1].clone()
        return out

    def optimizer_state(self) -> Dict[str, torch.Tensor]:
        """The optimizer's own state on the LOCAL ps shards (slots under their TF names, Adam's beta powers): the part of
        :meth:`state_dict` that is not a graph variable.  Kept across a fabric re-formation by the ps service."""
        sd = self.state_dict()
        return {k: v for k, v in sd.items() if "/" in k or k in ("beta1_power", "beta2_power")}

    def load_optimizer_state(self, state: Dict[str, torch.Tensor]) -> List[str]:
        """Write slots / beta powers saved by :meth:`optimizer_state` back into the local shards (names of other shards and
        shape mismatches are skipped).  Returns the names restored."""
        done: List[str] = []
        suffix = {"Momentum": "slot_m", "Adam": "slot_m", "Adam_1": "slot_v"}
        for r, rk in self.ranks.items():
            if r not in self.ps_ranks:
                continue
            s = self.ps_ranks.index(r)
            on_gpu = getattr(rk.device, "type", None) == "cuda"
            with (torch.cuda.device(rk.device) if on_gpu else contextlib.nullcontext()), \
                    (torch.cuda.stream(rk.stream) if on_gpu else contextlib.nullcontext()):
                for key, val in state.items():
                    if "/" not in key:
                        continue
                    name, slot = key.rsplit("/", 1)
                    lay = self.layout.get(name)
                    if lay is None or lay.shard != s or slot not in suffix or tuple(val.shape) != tuple(lay.shape):
                        continue
                    # (a pitched view: write through it, a reshape would copy)
                    self._var_view(rk, suffix[slot], lay).copy_(val.to(rk.device).float().reshape(lay.rows, lay.cols))
                    done.append(key)
                if s == 0 and self.kind == 2 and "beta1_power" in state and "beta2_power" in state:
                    b = rk.bufs["ctl0"].tensor(torch.float32, self.off["beta1_power"], 2)
                    b[0], b[1] = float(state["beta1_power"]), float(state["beta2_power"])
                    done += ["beta1_power", "beta2_power"]
            rk.sync()
        return done

    def read_ctl(self, shard: int, fld: str, count: int = 1):
        r = self.ps_ranks[shard]
        rk = self.ranks[r]
        rk.sync()
        t = rk.bufs["ctl%d" % shard].tensor(torch.int64, self.off[fld], count).cpu()
        return int(t[0]) if count == 1 else t.tolist()

    def step_stats(self) -> List[Dict[str, Any]]:
        """Device-side trace of the LOCAL ranks (SURVEY A19 on the fabric tier; the reference traces the whole step per task,
        example_in_graph.py:65-68).  ps shards: every ``ps_apply`` launch stamps ``(kind, %globaltimer at entry, %globaltimer
        when the tokens were released, global_step)`` into a ring in ps HBM (``trace_cap`` entries).  Workers (one-kernel
        step): CTA 0 of every ``mlp_step_kernel`` launch writes ``(kind, entry, token acquired, forward GEMM done, head done,
        exit, step, G)`` into the worker's ring (``worker_trace_cap`` rows) -- four phases per step.  Returns timeline events
        -- feed them to ``dtf.timeline.Timeline(step_stats=...)`` for a chrome trace with one process per
        ``/job:ps/task:k`` and ``/job:worker/task:i`` GPU; %globaltimer is one clock per GPU, synchronised across the box
        well enough (sub-microsecond) to read the ps and worker rows against each other."""
        from ..utils.timeline import events_from_ring
        events: List[Dict[str, Any]] = []
        for r, rk in self.ranks.items():
            if r in self.worker_ranks and self.tf32:
                w = self.worker_ranks.index(r)
                rk.stream.synchronize()
                rows = rk.bufs["stepring_w%d" % w].tensor(torch.int64, 0, (self.cfg.worker_trace_cap + 1) * 8).view(-1, 8).cpu().tolist()
                task = "/job:worker/task:%d" % w
                for kind, t_in, t_tok, t_fwd, t_head, t_out, step, _g in rows:
                    if kind == 0:
                        continue
                    name = {2: "mlp_step", 3: "mlp_forward"}.get(int(kind), "k%d" % kind)
                    phases = [(name + "/wait_token", t_in, t_tok), (name + "/forward_gemm", t_tok, t_fwd),
                              (name + "/head_softmax_xent", t_fwd, t_head), (name + "/backward_gemm_push", t_head, t_out)]
                    ring = [(10 + i, a, b, step) for i, (_, a, b) in enumerate(phases) if a and b]
                    events += events_from_ring(task, ring, {10 + i: ph[0] for i, ph in enumerate(phases)},
                                               gpu_index=rk.device.index or 0)
            if r not in self.ps_ranks:
                continue
            s = self.ps_ranks.index(r)
            rk.stream.synchronize()
            ring = rk.bufs["trace%d" % s].tensor(torch.int64, 0, self.cfg.trace_cap * 4).view(-1, 4).cpu().tolist()
            events += events_from_ring("/job:ps/task:%d" % s, [row for row in ring if row[0] != 0], {1: "ps_apply"},
                                       gpu_index=rk.device.index or 0)
        return sorted(events, key=lambda e: e["start_us"])

    def staleness(self, shard: int = 0) -> Dict[str, Any]:
        hist = self.read_ctl(shard, "staleness_hist", 16)
        tot = sum(hist)
        return {"hist": hist, "mean": (self.read_ctl(shard, "staleness_sum") / tot) if tot else 0.0, "count": tot}

    # ------------------------------------------------------------------------------------------------
    # launch descriptors (built once; per step only wait targets / data pointers change)
    # ------------------------------------------------------------------------------------------------
    def _build_launches(self) -> None:
        spec, cfg, lay = self.spec, self.cfg, self.layout
        B, D, H, C = spec.batch, spec.in_dim, spec.hidden, spec.classes
        self._w: Dict[int, Dict[str, Any]] = {}
        for r, rk in self.ranks.items():
            if r not in self.worker_ranks:
                continue
            w = self.worker_ranks.index(r)
            ldh = round_up(H, 8)
            misc = rk.bufs["misc_w%d" % w]
            # misc layout: [0..64) per-CTA loss partials f32 | [64] step counter u64 | [72] err u32 | [4096..] loss ring
            d: Dict[str, Any] = {"ldh": ldh, "loss_ptr": misc.ptr, "stepctr_ptr": misc.ptr + 64, "err_ptr": misc.ptr + 72,
                                 "hist_ptr": misc.ptr + 4096}
            mb = rk.bufs["mailbox_w%d" % w]
            d["mb0"] = mb.ptr

            def src(base: str, l: VarLayout, es: int) -> int:
                if (cfg.publish_replicas or self.nvls) and base == "shadow":
                    return rk.bufs["replica%d_w%d" % (l.shard, w)].ptr + l.offset * es      # local copy
                return self.peer[(r, "%s%d" % (base, l.shard))].ptr + l.offset * es

            def slot(l: VarLayout) -> int:
                if self.nvls:
                    return self.sym_grads[l.shard].local(r).ptr + l.offset * 4              # gradients stay local
                return self.peer[(r, "grads%d" % l.shard)].ptr + (w * self.shard_elems[l.shard] + l.offset) * 4

            def ctl_arrivals(shard: int) -> int:
                return self.peer[(r, "ctl%d" % shard)].ptr + self.off["w"] + w * self.off["w_stride"]

            x16 = rk.bufs["x16_w%d" % w]
            # ---- F1: h = relu(x . W1 + b1), W1 pulled from the ps inside the GEMM --------------------
            g1 = GemmArgs()
            g1.a, g1.lda = x16.ptr, D
            g1.b, g1.ldb = src("shadow", lay["hid_w"], 2), lay["hid_w"].pitch
            g1.c, g1.ldc, g1.c_bf16 = rk.bufs["h_w%d" % w].ptr, ldh, 1
            g1.M, g1.N, g1.K = B, H, D
            g1.a_mn, g1.b_mn = 0, 1
            g1.bias, g1.relu = src("master", lay["hid_b"], 4), 1
            g1.alpha, g1.splits = 1.0, 1
            g1.wait_flag = mb.ptr + lay["hid_w"].shard * self.mb_bytes      # token of the shard that owns W1
            g1.err, g1.timeout_ns = d["err_ptr"], cfg.timeout_ns
            g1.block_n_override = self.block_n_f1
            if cfg.f1_splits > 1:
                # split-K: several CTAs stream disjoint K ranges of x / W1 and red.add fp32 partials; bias + ReLU
                # move into the head, which also clears the accumulator for the next step
                g1.c, g1.ldc, g1.c_bf16 = rk.bufs["hacc_w%d" % w].ptr, ldh, 0
                g1.bias, g1.relu, g1.splits = None, 0, cfg.f1_splits
            d["g1"] = g1
            # ---- head ---------------------------------------------------------------------------------
            hd = MlpHeadArgs()
            hd.h, hd.ldh = rk.bufs["h_w%d" % w].ptr, ldh
            hd.w2, hd.ldw2 = src("shadow", lay["sm_w"], 2), lay["sm_w"].pitch
            hd.b2 = src("master", lay["sm_b"], 4)
            hd.labels, hd.ldl = rk.bufs["labels_w%d" % w].ptr, C
            hd.B, hd.H, hd.C, hd.clip_min = B, H, C, cfg.clip_min
            hd.loss_out, hd.loss_hist, hd.step_counter, hd.hist_cap = d["loss_ptr"], d["hist_ptr"], d["stepctr_ptr"], cfg.loss_hist
            hd.dh, hd.lddh = rk.bufs["dh_w%d" % w].ptr, ldh
            hd.gw2, hd.ldgw2 = slot(lay["sm_w"]), lay["sm_w"].pitch
            hd.gb2, hd.gb1 = slot(lay["sm_b"]), slot(lay["hid_b"])
            hd.mailbox = mb.ptr
            hd.rank, hd.stamp_from_version = w, 0 if cfg.sync else 1
            hd.sys_scope = 0 if cfg.colocated else 1
            hd.ctas = self.head_ctas
            if cfg.f1_splits > 1:
                hd.h_acc, hd.ld_acc, hd.b1 = rk.bufs["hacc_w%d" % w].ptr, ldh, src("master", lay["hid_b"], 4)
            d["head"] = hd
            # Shards the head pushes to.  The dW1 GEMM (same stream, later) signals the shard that owns hid_w
            # on behalf of the whole push: kernel-boundary ordering makes the head's stores visible first.
            head_shards = sorted({lay["sm_w"].shard, lay["sm_b"].shard, lay["hid_b"].shard} - {lay["hid_w"].shard})
            d["head_ctls"] = [self.peer[(r, "ctl%d" % s)].ptr for s in head_shards]
            d["head_mailboxes"] = [mb.ptr + s * self.mb_bytes for s in head_shards]
            # ---- B3: dW1 = x^T . dh pushed into the ps slot ------------------------------------------
            g3 = GemmArgs()
            g3.a, g3.lda = x16.ptr, D
            g3.b, g3.ldb = rk.bufs["dh_w%d" % w].ptr, ldh
            g3.c, g3.ldc, g3.c_bf16 = slot(lay["hid_w"]), lay["hid_w"].pitch, 0
            g3.M, g3.N, g3.K = D, H, B
            g3.a_mn, g3.b_mn = 1, 1
            g3.alpha, g3.splits = 1.0, 1
            g3.signal = ctl_arrivals(lay["hid_w"].shard)
            g3.signal_gpu_scope = 1 if cfg.colocated else 0
            # the GEMM's first CTA also publishes the stamp (local_step / pulled version) for this push
            g3.stamp_src = mb.ptr + lay["hid_w"].shard * self.mb_bytes + (0 if cfg.sync else 8)
            g3.stamp_dst = ctl_arrivals(lay["hid_w"].shard) + 8
            g3.block_n_override = self.block_n_b3
            d["g3"] = g3
            d["extra_wait_shards"] = [s for s in range(cfg.num_ps) if s != lay["hid_w"].shard]
            if self.tf32:
                # ---- the whole step as one kernel (csrc/mlp_step.cu): fp32 parameters read in place ------------------
                def psrc(l: VarLayout, r=r, rk=rk, w=w) -> int:
                    if self.nvls:
                        return rk.bufs["replica%d_w%d" % (l.shard, w)].ptr + l.offset * 4       # local fp32 replica
                    return self.peer[(r, "master%d" % l.shard)].ptr + l.offset * 4              # the ps's master (same GPU / NVLink)

                # everything the argument block points at, resolved NOW (the builder below is called later, from
                # attach_dataset / evaluate / the plan builder, when this loop's variables have moved on)
                d["step_const"] = dict(
                    w=w, w1=psrc(lay["hid_w"]), ldw1=lay["hid_w"].pitch, b1=psrc(lay["hid_b"]),
                    w2=psrc(lay["sm_w"]), ldw2=lay["sm_w"].pitch, b2=psrc(lay["sm_b"]),
                    scr=rk.bufs["stepscr_w%d" % w].ptr, flags=rk.bufs["stepflags_w%d" % w].ptr,
                    ring=rk.bufs["stepring_w%d" % w].ptr,
                    gw1=slot(lay["hid_w"]), gb1=slot(lay["hid_b"]), gw2=slot(lay["sm_w"]), gb2=slot(lay["sm_b"]),
                    tokens=[(rk.bufs["replica%d_w%d" % (sh, w)].ptr + self.shard_elems[sh] * 4) if self._mc_tokens()
                            else (mb.ptr + sh * self.mb_bytes) for sh in self.var_shards],
                    token_scale=[int(self.lib.dtf_ps_apply_grid(self.shard_elems[sh])) if self._mc_tokens() else 1
                                 for sh in self.var_shards],
                    mb_tokens=[mb.ptr + sh * self.mb_bytes for sh in self.var_shards],
                    arrivals=[ctl_arrivals(sh) for sh in self.var_shards],
                    consumed=[self.peer[(r, "ctl%d" % sh)].ptr + self.off["consumed"] + w * 8 for sh in self.var_shards])
                d["step_staged"] = self._step_args(d, rk.bufs["xf32_w%d" % w].ptr, 128, rk.bufs["labels_w%d" % w].ptr)
            self._w[r] = d
        self._p: Dict[int, PsApplyArgs] = {}
        for r, rk in self.ranks.items():
            if r not in self.ps_ranks:
                continue
            s = self.ps_ranks.index(r)
            n = self.shard_elems[s]
            a = PsApplyArgs()
            a.ctl, a.master = rk.bufs["ctl%d" % s].ptr, rk.bufs["master%d" % s].ptr
            a.slot_m, a.slot_v = rk.bufs["slot_m%d" % s].ptr, rk.bufs["slot_v%d" % s].ptr
            a.shadow = rk.bufs["shadow%d" % s].ptr
            for w in range(cfg.num_workers):
                a.grad[w] = self.peer[(r, "sgrads%d_w%d" % (s, w))].ptr if self.nvls else rk.bufs["grads%d" % s].ptr + w * n * 4
                a.mailbox[w] = self.peer[(r, "mailbox_w%d" % w)].ptr + s * self.mb_bytes
                if (cfg.publish_replicas or (self.nvls and not self.nvls_multicast)) and not self.tf32:
                    a.replica[w] = self.peer[(r, "replica%d_w%d" % (s, w))].ptr
            if self.tf32:
                a.shadow = None                                  # no bf16 copy: the fp32 master (or its multicast replica) is the pull source
            if self.nvls and self.nvls_multicast:
                a.grad_mc = self.sym_grads[s].mc(r)
                if self.tf32:
                    a.master_mc = self.sym_repl[s].mc(r)         # ONE multimem.st of fp32 parameters into every GPU's replica
                    if self._mc_tokens():
                        a.token_mc = self.sym_repl[s].mc(r) + n * 4
                else:
                    a.shadow_mc = self.sym_repl[s].mc(r)
            a.n, a.num_workers, a.replicas_to_aggregate = n, cfg.num_workers, self.R
            a.ctas_per_push = self.ctas_per_push[s]
            a.mode, a.kind = (0 if cfg.sync else 1), self.kind
            a.lr = float(self.opt["lr"])
            a.momentum = float(self.opt.get("momentum", 0.0))
            a.beta1, a.beta2, a.eps = float(self.opt.get("beta1", 0.9)), float(self.opt.get("beta2", 0.999)), \
                float(self.opt.get("eps", self.opt.get("epsilon", 1e-8)))
            a.nesterov = int(bool(self.opt.get("nesterov", False)))
            a.publish_replicas = int((cfg.publish_replicas or (self.nvls and not self.nvls_multicast)) and not self.tf32)
            a.num_zero = 0
            if self.head_ctas > 1 or self.tf32:
                # the row-parallel head accumulates dW2 / db2 / db1 with atomics: clear those slot ranges after reading
                for vn in ("sm_w", "sm_b", "hid_b"):
                    l = lay[vn]
                    if l.shard == s:
                        a.zero_begin[a.num_zero], a.zero_end[a.num_zero] = l.offset, l.offset + l.numel_padded
                        a.num_zero += 1
            a.timeout_ns = cfg.timeout_ns
            a.trace, a.trace_cap = rk.bufs["trace%d" % s].ptr, cfg.trace_cap
            a.grid = 0
            a.system_scope = 0 if cfg.colocated else 1
            self._p[r] = a

    def _mc_tokens(self) -> bool:
        """Workers wait on a counter in their own replica buffer that every ps_apply CTA bumps through the switch
        (multimem.red) right after its release fence -- no last-block round -- when: tf32 engine, NVLS multicast, sync with
        replicas_to_aggregate == total replicas (a token for every replica after every aggregate)."""
        return bool(self.tf32 and self.nvls and self.nvls_multicast and self.cfg.sync and self.R == self.cfg.num_workers
                    and os.environ.get("DTF_MC_TOKENS", "1") == "1")

    def _step_args(self, d: Dict[str, Any], x_ptr: int, x_rows: int, lab_ptr: int, nbatches: int = 0,
                   rows: Optional[int] = None) -> MlpStepArgs:
        """Argument block of ``dtf_mlp_step`` for one worker: ``x`` / labels = a staged batch (``nbatches == 0``) or a
        device-resident dataset walked by the device step counter."""
        spec, cfg, lay, k = self.spec, self.cfg, self.layout, d["step_const"]
        a = MlpStepArgs()
        a.B, a.D, a.H, a.C, a.G, a.phase_mask = (rows or spec.batch), spec.in_dim, spec.hidden, spec.classes, self.step_ctas, 7
        a.x, a.ldx, a.x_rows = x_ptr, spec.in_dim, x_rows
        a.labels, a.ldl = lab_ptr, spec.classes
        a.nbatches, a.bstride, a.boffset = nbatches, cfg.num_workers, k["w"]
        a.w1, a.ldw1, a.b1 = k["w1"], k["ldw1"], k["b1"]
        a.w2, a.ldw2, a.b2 = k["w2"], k["ldw2"], k["b2"]
        a.hpart, a.dh, a.lddh = k["scr"], k["scr"] + self.step_ctas * 128 * (round_up(spec.hidden, 16) + 4) * 4, 128
        a.head_part = a.dh + (128 * 128 + 64) * 4
        a.flags = k["flags"]
        a.gw1, a.ldgw1, a.gb1 = k["gw1"], lay["hid_w"].pitch, k["gb1"]
        a.gw2, a.ldgw2, a.gb2 = k["gw2"], lay["sm_w"].pitch, k["gb2"]
        a.clip_min, a.loss_out, a.step_counter = cfg.clip_min, d["loss_ptr"], d["stepctr_ptr"]
        a.num_tokens = a.num_signals = len(self.var_shards)
        for i in range(len(self.var_shards)):
            a.token[i] = k["tokens"][i]
            a.token_scale[i] = k["token_scale"][i]
            a.token_base[i] = d.get("token_base", [0, 0, 0, 0])[i]
            if cfg.sync and self.R < cfg.num_workers:
                a.consumed[i] = k["consumed"][i]           # backup workers: never overwrite a push the ps has not consumed / dropped
            a.arrivals[i] = k["arrivals"][i]
            # the stamp (which parameters this push was computed from) is what the ps's staleness / stale-gradient logic
            # reads; with replicas_to_aggregate == replicas every aggregate is all-fresh by construction and the ps never
            # looks at it (ps_engine.cu all_fresh_only) -- skipping the remote store there also takes a pending NVLink
            # write out from under the step kernel's release fence
            a.stamp_dst[i] = 0 if (cfg.sync and self.R == cfg.num_workers and os.environ.get("DTF_STAMP_ALWAYS", "0") != "1") \
                else k["arrivals"][i] + 8
            a.stamp_src[i] = k["mb_tokens"][i] + (0 if cfg.sync else 8)   # token (sync) / pulled version (async)
        # sync: the push is stamped with the token the worker holds (= global step at the pull); with the multicast counter
        # tokens the mailbox token may lag one aggregate, and step == global step there (all-fresh aggregates only)
        a.stamp_step = 1 if (cfg.sync and self._mc_tokens()) else 0
        a.sys_scope = 0 if cfg.colocated else 1
        a.timeout_ns, a.err = cfg.timeout_ns, d["err_ptr"]
        a.no_cluster = int(os.environ.get("DTF_STEP_NO_CLUSTER", "0") == "1")
        a.dbg = int(os.environ.get("DTF_STEP_DBG", "0"))
        a.ring, a.ring_cap = k["ring"], cfg.worker_trace_cap
        return a

    # ------------------------------------------------------------------------------------------------
    # stepping
    # ------------------------------------------------------------------------------------------------
    def launches_per_worker_step(self, source: str = "staged") -> int:
        if self.tf32:
            return 1
        any_w = next(iter(self._w.values()), None)
        extra = len(any_w["extra_wait_shards"]) if any_w else 0
        nhead = len(any_w["head_ctls"]) if any_w else 0
        return 3 + extra + max(nhead - 1, 0) + (1 if source == "dataset" else 0)

    def attach_dataset(self, rank: int, images, labels) -> None:
        """Stage a whole split in this worker's HBM (fp32 images [N, in_dim], one-hot labels [N, classes]).
        Worker ``w`` of ``W`` then walks batches ``w, w+W, w+2W, ...`` (mod the number of batches): the batch
        index is computed ON THE DEVICE from the step counter, so steps are CUDA-graph replayable."""
        rk, d = self.ranks[rank], self._w[rank]
        B = self.spec.batch
        with torch.cuda.device(rk.device):
            img = torch.as_tensor(images, dtype=torch.float32).contiguous().to(rk.device)
            lab = torch.as_tensor(labels, dtype=torch.float32).contiguous().to(rk.device)
        d["ds_images"], d["ds_labels"], d["ds_nbatches"] = img, lab, img.shape[0] // B
        assert d["ds_nbatches"] >= 1
        if self.tf32:
            # the step kernel's TMA reads the batch straight out of the dataset (row = batch index x B, from the device step
            # counter): no staging pass at all
            d["step_ds"] = self._step_args(d, img.data_ptr(), img.shape[0], lab.data_ptr(), d["ds_nbatches"])

    def enqueue_worker_step(self, rank: int, source: str = "staged") -> None:
        """Enqueue one worker step on the rank's stream.  ``source='staged'``: the batch is already in the
        rank's staging buffers (see :meth:`stage_batch`); ``'dataset'``: take the next batch of the attached
        device-resident dataset (one extra staging kernel).  Wait targets come from the device step counter."""
        rk, d = self.ranks[rank], self._w[rank]
        st = rk.stream.cuda_stream
        lib = self.lib
        w = self.worker_ranks.index(rank)
        n = 0
        if self.tf32:
            a = d["step_ds"] if source == "dataset" else d["step_staged"]
            with torch.cuda.device(rk.device):
                rc = lib.dtf_mlp_step(ctypes.byref(a), st)
            assert rc == 0, "mlp_step rc=%d" % rc
            cuda_lib._bump(1)
            rk.step += 1
            self._last_step_launches = 1
            return
        with torch.cuda.device(rk.device):
            def stage_next():
                rc_ = lib.dtf_stage_from_dataset(d["ds_images"].data_ptr(), d["ds_labels"].data_ptr(), d["ds_nbatches"],
                                                 self.spec.batch, self.spec.in_dim, self.spec.classes,
                                                 self.cfg.num_workers, w, d["stepctr_ptr"],
                                                 rk.bufs["x16_w%d" % w].ptr, rk.bufs["labels_w%d" % w].ptr, st)
                assert rc_ == 0, "stage_from_dataset rc=%d" % rc_
            if source == "dataset" and not d.get("primed"):
                stage_next()             # first batch; afterwards each step stages its successor's batch at its END,
                d["primed"] = True       # i.e. while the ps is aggregating (the worker would otherwise just wait)
                n += 1
            for s in d["extra_wait_shards"]:
                rc = lib.dtf_wait_token(rk.bufs["mailbox_w%d" % w].ptr + s * self.mb_bytes, 0, d["stepctr_ptr"],
                                        self.cfg.timeout_ns, d["err_ptr"], st)
                assert rc == 0, rc
                n += 1
            if self.cfg.sync and self.R < self.cfg.num_workers:
                # backup workers: the slot is rewritten only once the ps consumed or dropped this worker's previous push
                for s in range(self.cfg.num_ps):
                    if self.ctas_per_push[s]:
                        rc = lib.dtf_wait_token(self.peer[(rank, "ctl%d" % s)].ptr + self.off["consumed"] + w * 8,
                                                rk.step * self.ctas_per_push[s], None, self.cfg.timeout_ns, d["err_ptr"], st)
                        assert rc == 0, rc
                        n += 1
            g1, hd, g3 = d["g1"], d["head"], d["g3"]
            g1.wait_target, g1.wait_target_ptr = 0, d["stepctr_ptr"]
            rc = lib.dtf_gemm_bf16(ctypes.byref(g1), st)
            assert rc == 0, "F1 gemm rc=%d" % rc
            # the head signals the first shard it ALONE pushed to (if any); further such shards get a
            # signal-only launch; the shard owning hid_w is signalled by the dW1 GEMM for the whole push
            if d["head_ctls"]:
                hd.ctl, hd.mailbox = d["head_ctls"][0], d["head_mailboxes"][0]
            else:
                hd.ctl, hd.mailbox = None, d["mb0"]
            rc = lib.dtf_mlp_head(ctypes.byref(hd), st)
            assert rc == 0, "mlp_head rc=%d" % rc
            n += 2
            for ctl_ptr, mbp in zip(d["head_ctls"][1:], d["head_mailboxes"][1:]):
                rc = lib.dtf_push_grad(0, 0, 0, ctl_ptr, mbp, w, hd.stamp_from_version, 1, 1, st)
                assert rc == 0, rc
                n += 1
            rc = lib.dtf_gemm_bf16(ctypes.byref(g3), st)
            assert rc == 0, "B3 gemm rc=%d" % rc
            n += 1
            if source == "dataset":
                stage_next()             # reads the step counter the head just advanced -> batch of step t+1
                n += 1
        cuda_lib._bump(n)
        rk.step += 1
        self._last_step_launches = n

    # -- the interface the graph-API strategy drives (same shape as GenericPSEngine's) ------------------------------------
    def prepare(self) -> None:
        self.init_params()

    def ps_apply(self, rank: int, idle_ok: bool = False) -> None:
        """One apply launch of the local ps shard; ``idle_ok``: a timed-out wait for pushes is not an error (service loop)."""
        a = self._p[rank]
        a.idle_ok = int(idle_ok)
        # a service loop polls: short waits (no push yet = not an error), so that host-side requests -- stop, farewell -- are
        # seen within milliseconds
        a.timeout_ns = min(int(self.cfg.timeout_ns), 50_000_000) if idle_ok else int(self.cfg.timeout_ns)
        self.enqueue_ps_apply(rank)

    def release_all_tokens(self, rank: int) -> None:
        """End of training (a sync replica left): write a token no step will ever exceed into every worker's mailbox for the
        LOCAL ps shard, so a replica blocked in its device-side token wait completes the step it is in."""
        rk = self.ranks[rank]
        s = self.ps_ranks.index(rank)
        rk.sync()
        with torch.cuda.device(rk.device):
            for w in range(self.cfg.num_workers):
                self.peer[(rank, "mailbox_w%d" % w)].tensor(torch.int64, s * self.mb_bytes, 2).fill_(1 << 62)
            torch.cuda.synchronize(rk.device)

    def adopt_global_step(self, rank: int) -> int:
        """Worker ``rank``: take each ps shard's CURRENT global step as the base of its token sequence -- a run restored from
        a checkpoint, or a fabric re-formed after a task failure, starts with ``global_step`` = g on the ps while this
        worker's device step counter starts at 0.  Sync: its mailbox token / version become g (as if the ps had just handed
        it the token of step g) and step k waits for token >= g + k; async tokens are push COUNTS and need no base.  Call
        before the first step (the step plans copy the argument block).  Returns shard 0's global step."""
        rk, d = self.ranks[rank], self._w[rank]
        w = self.worker_ranks.index(rank)
        rk.sync()
        base, mb = [0, 0, 0, 0], rk.bufs["mailbox_w%d" % w]
        out = 0
        with torch.cuda.device(rk.device):
            for i, sh in enumerate(self.var_shards):
                gs = int(self.peer[(rank, "ctl%d" % sh)].tensor(torch.int64, self.off["global_step"], 1).cpu()[0])
                if i == 0 or sh == 0:
                    out = gs                                                         # shard 0 owns the graph's global_step
                mb.tensor(torch.int64, sh * self.mb_bytes, 2).fill_(gs)             # {token, version}
                if self.cfg.sync and not self._mc_tokens():
                    base[i] = gs
                elif not self.cfg.sync:
                    mb.tensor(torch.int64, sh * self.mb_bytes, 1).fill_(0)          # async: token = applied-push count
            torch.cuda.synchronize(rk.device)
        d["token_base"] = base
        if self.tf32:
            d["step_staged"] = self._step_args(d, rk.bufs["xf32_w%d" % w].ptr, 128, rk.bufs["labels_w%d" % w].ptr)
        return out

    def var_tensor(self, rank: int, name: str) -> torch.Tensor:
        """True-shape fp32 view of variable ``name`` in the LOCAL ps shard's master buffer (graph variables are bound to it)."""
        return self._var_view(self.ranks[rank], "master", self.layout[name])

    def global_step_tensor(self, rank: int) -> torch.Tensor:
        return self.ranks[rank].bufs["ctl0"].tensor(torch.int64, self.off["global_step"], 1).view(())

    def enqueue_ps_apply(self, rank: int) -> None:
        rk = self.ranks[rank]
        with torch.cuda.device(rk.device):
            rc = self.lib.dtf_ps_apply(ctypes.byref(self._p[rank]), (rk.ps_stream or rk.stream).cuda_stream)
        assert rc == 0, "ps_apply rc=%d" % rc
        cuda_lib._bump()

    def stage_batch(self, rank: int, x: torch.Tensor, y: torch.Tensor) -> None:
        """Host (pinned) or device fp32 batch -> the rank's bf16/f32 staging buffers, on the rank's stream."""
        rk = self.ranks[rank]
        w = self.worker_ranks.index(rank)
        B, D, C = self.spec.batch, self.spec.in_dim, self.spec.classes
        with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
            xf = rk.bufs["xf32_w%d" % w].tensor(torch.float32, 0, B * D).view(B, D)
            xf.copy_(x, non_blocking=True)
            rk.bufs["labels_w%d" % w].tensor(torch.float32, 0, B * C).view(B, C).copy_(y, non_blocking=True)
            if self.tf32:
                return                    # the step kernel reads the fp32 staging buffer in place
            rc = self.lib.dtf_convert_f32_bf16(xf.data_ptr(), D, rk.bufs["x16_w%d" % w].ptr, D, B, D, D,
                                               rk.stream.cuda_stream)
            assert rc == 0, rc
        cuda_lib._bump()

    # ------------------------------------------------------------------------------------------------
    # native step plans (end-to-end path: one C call per rank per step, see csrc/step_exec.cu)
    # ------------------------------------------------------------------------------------------------
    def _plans(self) -> Dict[str, Any]:
        """Per-rank op sequences for ``step(x_pinned, y_pinned)``.  Input staging is DOUBLE-BUFFERED and runs on a
        copy stream: ``copy[p]`` = wait until the compute stream is done with buffer set ``p`` -> H2D x -> H2D y ->
        fp32->bf16 staging kernel -> record ``ready[p]``; ``compute[p]`` = wait ``ready[p]`` -> the worker's
        kernels on buffer set ``p`` (-> the ps's apply kernels when colocated) -> record ``done[p]``.  A step
        alternates ``p``; ``step(..., prefetch=(x_next, y_next))`` issues ``copy[p^1]`` for the NEXT batch right
        after launching this step's kernels, so the PCIe transfer overlaps the step's compute.  The rank whose loss
        is returned adds D2H of the loss partials into pinned host memory + a stream sync.  Built once; per step
        only the H2D source pointers change."""
        got = getattr(self, "_native_plans", None)
        if got is not None:
            return got
        from ..ops.cuda_lib import (OP_CONVERT, OP_D2H, OP_GEMM, OP_H2D, OP_HEAD, OP_MLP_STEP, OP_PS_APPLY, OP_SIGNAL, OP_SYNC,
                                    OP_WAIT_TOKEN, StepOp, StepPlan)
        OP_EVENT_RECORD, OP_EVENT_WAIT = 11, 12
        B, D, C = self.spec.batch, self.spec.in_dim, self.spec.classes
        plans: Dict[str, Any] = {"copy": {}, "compute": {}, "ps": {}, "loss": {}, "loss_async": {}, "pending": {}, "keep": []}
        for r, rk in self.ranks.items():
            st = rk.stream.cuda_stream
            if r in self.worker_ranks:
                w = self.worker_ranks.index(r)
                d = self._w[r]
                with torch.cuda.device(rk.device):
                    copy_stream = torch.cuda.Stream(rk.device)
                    events = []
                    for _ in range(4):                       # ready[0], ready[1], done[0], done[1]
                        ev = torch.cuda.Event()
                        ev.record(rk.stream)                 # materialises the cudaEvent_t (and makes the first wait a no-op)
                        events.append(ev)
                plans["keep"] += [copy_stream] + events
                ready, done = events[:2], events[2:]
                g1, hd, g3 = d["g1"], d["head"], d["g3"]
                g1.wait_target, g1.wait_target_ptr = 0, d["stepctr_ptr"]
                if d["head_ctls"]:
                    hd.ctl, hd.mailbox = d["head_ctls"][0], d["head_mailboxes"][0]
                else:
                    hd.ctl, hd.mailbox = None, d["mb0"]
                plans["copy"][r], plans["compute"][r] = [], []
                for par in range(2):
                    sfx = "" if par == 0 else "b"
                    if par == 1:
                        for base, nbytes in (("xf32", 128 * D * 4), ("labels", 128 * 16 * 4), ("x16", 128 * D * 2)):
                            name = "%sb_w%d" % (base, w)
                            if name not in rk.bufs:
                                rk.bufs[name] = self.fabric.alloc(r, name, nbytes)
                    xf = rk.bufs["xf32%s_w%d" % (sfx, w)].ptr
                    lab = rk.bufs["labels%s_w%d" % (sfx, w)].ptr
                    x16 = rk.bufs["x16%s_w%d" % (sfx, w)].ptr
                    if par == 0:
                        g1p, hdp, g3p = g1, hd, g3
                    else:
                        g1p, hdp, g3p = type(g1).from_buffer_copy(g1), type(hd).from_buffer_copy(hd), type(g3).from_buffer_copy(g3)
                        g1p.a, g3p.a, hdp.labels = x16, x16, lab
                    cops = [StepOp(kind=OP_EVENT_WAIT, p0=done[par].cuda_event),
                            StepOp(kind=OP_H2D, p0=xf, p1=None, i0=B * D * 4), StepOp(kind=OP_H2D, p0=lab, p1=None, i0=B * C * 4)]
                    if not self.tf32:
                        cops.append(StepOp(kind=OP_CONVERT, p0=xf, p1=x16, i0=D, i1=D, i2=B, i3=D, i4=D))
                    cops.append(StepOp(kind=OP_EVENT_RECORD, p0=ready[par].cuda_event))
                    plans["copy"][r].append(StepPlan(cops, rk.device.index, copy_stream.cuda_stream))
                    ops = [StepOp(kind=OP_EVENT_WAIT, p0=ready[par].cuda_event)]
                    if self.tf32:
                        # fp32 staging buffer read in place by the step kernel's TMA: H2D -> ONE kernel -> (ps apply)
                        sp = d["step_staged"] if par == 0 else self._step_args(d, xf, 128, lab)
                        ops.append(StepOp(kind=OP_MLP_STEP, p0=ctypes.addressof(sp)))
                        keep = [sp]
                    else:
                        for s_ in d["extra_wait_shards"]:
                            ops.append(StepOp(kind=OP_WAIT_TOKEN, p0=rk.bufs["mailbox_w%d" % w].ptr + s_ * self.mb_bytes,
                                              p1=d["stepctr_ptr"], p2=d["err_ptr"], i0=0, u0=self.cfg.timeout_ns))
                        ops.append(StepOp(kind=OP_GEMM, p0=ctypes.addressof(g1p)))
                        ops.append(StepOp(kind=OP_HEAD, p0=ctypes.addressof(hdp)))
                        for ctl_ptr, mbp in zip(d["head_ctls"][1:], d["head_mailboxes"][1:]):
                            ops.append(StepOp(kind=OP_SIGNAL, p0=ctl_ptr, p1=mbp, i0=w, i1=hd.stamp_from_version))
                        ops.append(StepOp(kind=OP_GEMM, p0=ctypes.addressof(g3p)))
                        keep = [g1p, hdp, g3p]
                    if r in self.ps_ranks and rk.ps_stream is None:
                        # ps and worker share the GPU and the stream: the apply joins the worker's plan (one graph)
                        ops += [StepOp(kind=OP_PS_APPLY, p0=ctypes.addressof(self._p[r]))
                                for _ in range(1 if self.cfg.sync else self.cfg.num_workers)]
                        keep.append(self._p[r])
                    ops.append(StepOp(kind=OP_EVENT_RECORD, p0=done[par].cuda_event))
                    plans["compute"][r].append(StepPlan(ops, rk.device.index, st, keep=keep))
                host = torch.zeros(16, dtype=torch.float32).pin_memory()
                plans["loss"][r] = (StepPlan([StepOp(kind=OP_D2H, p0=host.data_ptr(), p1=d["loss_ptr"], i0=self.head_ctas * 4),
                                              StepOp(kind=OP_SYNC)], rk.device.index, st), host.numpy(), host)
            if r in self.ps_ranks and (r not in self.worker_ranks or rk.ps_stream is not None):
                k = 1 if self.cfg.sync else self.cfg.num_workers
                plans["ps"][r] = StepPlan([StepOp(kind=OP_PS_APPLY, p0=ctypes.addressof(self._p[r])) for _ in range(k)],
                                          rk.device.index, (rk.ps_stream or rk.stream).cuda_stream, keep=[self._p[r]])
        plans["runs"], plans["parity"], plans["prefetched"] = 0, 0, None
        self._native_plans = plans
        return plans

    def _loss_async_plans(self, r: int):
        """Deferred read-back of worker ``r``'s loss (built on first use): one pinned landing buffer + event per parity;
        the plan copies the head's loss partials D2H right behind the step's kernels and records the event behind the
        copy -- ``PendingLoss.result()`` waits on that event only."""
        plans = self._native_plans
        got = plans["loss_async"].get(r)
        if got is None:
            from ..ops.cuda_lib import OP_D2H, StepOp, StepPlan
            OP_EVENT_RECORD = 11
            rk, d = self.ranks[r], self._w[r]
            got = []
            for _ in range(2):
                hostp = torch.zeros(16, dtype=torch.float32).pin_memory()
                with torch.cuda.device(rk.device):
                    lev = torch.cuda.Event()
                    lev.record(rk.stream)        # materialises the cudaEvent_t
                lpl = StepPlan([StepOp(kind=OP_D2H, p0=hostp.data_ptr(), p1=d["loss_ptr"], i0=self.head_ctas * 4),
                                StepOp(kind=OP_EVENT_RECORD, p0=lev.cuda_event)], rk.device.index, rk.stream.cuda_stream)
                got.append((lpl, hostp.numpy(), hostp, lev))
            plans["loss_async"][r] = got
        return got

    def _graph_plans(self) -> None:
        """After both buffer sets have run eagerly once: every kernel run of every compute / ps plan becomes ONE
        CUDA-graph launch, so a step costs the host two memcpy enqueues + a staging launch (copy stream) and one
        graph launch per worker (+ the loss read-back)."""
        plans = self._native_plans
        self.synchronize()
        for r in list(plans["compute"]):
            plans["compute"][r] = [pl.graphed() for pl in plans["compute"][r]]
        for r in list(plans["ps"]):
            plans["ps"][r] = plans["ps"][r].graphed()
        plans["graphed"] = True

    def _is_pinned_f32(self, t) -> bool:
        """Pinned contiguous fp32 host tensor?  (``is_pinned`` asks the driver: cache the answer per storage range.)"""
        if not isinstance(t, torch.Tensor) or t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            return False
        cache = self.__dict__.setdefault("_pinned_cache", {})
        key = (t.data_ptr(), t.numel())
        ok = cache.get(key)
        if ok is None:
            if len(cache) > 65536:
                cache.clear()
            ok = cache[key] = bool(t.is_pinned())
        return ok

    def _issue_copy(self, plans, local_workers, par: int, x: torch.Tensor, y: torch.Tensor) -> None:
        B = self.spec.batch
        split = len(local_workers) > 1 and x.shape[0] == B * len(local_workers)
        xp, yp = x.data_ptr(), y.data_ptr()
        xs, ys = B * self.spec.in_dim * 4, B * self.spec.classes * 4
        for i, r in enumerate(local_workers):
            pl = plans["copy"][r][par]
            pl.ops[1].p1 = xp + (i * xs if split else 0)
            pl.ops[2].p1 = yp + (i * ys if split else 0)
            pl.run()

    def step(self, x=None, y=None, sync_loss=True, source: str = "dataset", prefetch=None):
        """One training step for every LOCAL rank.  Workers: (optional staging of the host batch) +
        3 kernels; ps shards: one ps_apply per aggregate (sync) or per worker push (async).
        Returns the local worker's loss when ``sync_loss`` (a device->host read).  ``sync_loss="deferred"`` returns a
        :class:`PendingLoss` instead: the read-back is enqueued behind the step's kernels and ``.result()`` waits for
        it later -- call ``step`` for batch t+1 first and the host's turnaround overlaps step t on the GPU.

        ``x``/``y``: one batch ``[B, in_dim]`` / ``[B, classes]`` (every local worker trains on it) or, with several
        local workers (in-graph replication), ``[W_local * B, ...]`` split across them in worker order -- the
        scatter of ``example_in_graph.py:38``.  Pinned fp32 host tensors take the native path: ONE C call per rank
        and stream enqueues the H2D copies + staging kernel (copy stream) and the step's kernels, CUDA-graphed
        (``csrc/step_exec.cu``).  ``prefetch=(x_next, y_next)``: start the next step's host->device copy now, so it
        overlaps this step's kernels (input double buffering; the next ``step`` must be called with those tensors)."""
        cfg = self.cfg
        local_workers = [r for r in self.worker_ranks if r in self.ranks]
        if x is not None and self._is_pinned_f32(x) and self._is_pinned_f32(y):
            plans = self._plans()
            par = plans["parity"]
            if plans["prefetched"] != (x.data_ptr(), y.data_ptr(), par):
                self._issue_copy(plans, local_workers, par, x, y)
            plans["prefetched"] = None
            for r in local_workers:
                plans["compute"][r][par].run()
                self.ranks[r].step += 1
            for r in self.ps_ranks:
                if r in plans["ps"]:
                    plans["ps"][r].run()
            if prefetch is not None and self._is_pinned_f32(prefetch[0]) and self._is_pinned_f32(prefetch[1]):
                self._issue_copy(plans, local_workers, par ^ 1, prefetch[0], prefetch[1])
                plans["prefetched"] = (prefetch[0].data_ptr(), prefetch[1].data_ptr(), par ^ 1)
            plans["parity"] = par ^ 1
            plans["runs"] += 1
            if plans["runs"] == 4 and not plans.get("graphed") and os.environ.get("DTF_E2E_GRAPH", "1") == "1":
                self._graph_plans()
            if sync_loss == "deferred" and local_workers:
                lpl, host_np, _, lev = self._loss_async_plans(local_workers[0])[par]
                old = plans["pending"].get(par)
                if old is not None:
                    old.result()              # its landing buffer and event are about to be reused
                lpl.run()
                plans["pending"][par] = pending = PendingLoss(lev, host_np, self.head_ctas)
                return pending
            if sync_loss and local_workers:
                pl, host_np, _ = plans["loss"][local_workers[0]]
                pl.run()
                return float(host_np[:self.head_ctas].sum())
            return None
        for i, r in enumerate(local_workers):
            if x is not None:
                B = self.spec.batch
                if len(local_workers) > 1 and x.shape[0] == B * len(local_workers):
                    self.stage_batch(r, x[i * B:(i + 1) * B], y[i * B:(i + 1) * B])
                else:
                    self.stage_batch(r, x, y)
            self.enqueue_worker_step(r, "staged" if x is not None else source)
        for r in self.ps_ranks:
            if r in self.ranks:
                for _ in range(1 if cfg.sync else cfg.num_workers):
                    self.enqueue_ps_apply(r)
        if sync_loss == "deferred":
            return PendingLoss(None, None, 0, value=self.read_loss())
        if sync_loss:
            return self.read_loss()
        return None

    def train_loop(self, x_batches, y_batches, steps: int, first: int = 0, stride: int = 1, depth: int = 2, prefetch_next: bool = False):
        """``steps`` end-to-end training steps in ONE native call (``csrc/step_exec.cu: dtf_run_loop``) -- the reference's
        ``while`` loop around ``mon_sess.run([train_step, global_step, loss], feed_dict=...)``
        (``/root/reference/distributed_mnist.py:148-152``) without the interpreter between the steps.

        ``x_batches`` ``[nb, B, in_dim]`` / ``y_batches`` ``[nb, B, classes]``: pinned contiguous fp32 HOST tensors.  Step i
        trains on batch ``(first + i * stride) % nb``: every step its batch is copied host->device (copy stream, one step
        ahead of the kernels that consume it), the step runs (the same CUDA-graphed plans ``step()`` uses), and the step's
        loss partials are copied device->host into row i of a pinned array; the host stays at most ``depth`` steps ahead
        of the landed losses.  ``prefetch_next``: also start the copy of the batch after the last step, so that a following
        ``train_loop`` / ``step`` on that batch finds it on the device (one continuous loop across calls).  Returns the
        ``steps`` losses (numpy fp32).  One local worker per process (between-graph
        replication); other topologies, and a process whose plans are not built yet, take ``step()`` per step."""
        import numpy as np
        from ..ops.cuda_lib import LoopArgs
        B, D, C = self.spec.batch, self.spec.in_dim, self.spec.classes
        steps = int(steps)
        local_workers = [r for r in self.worker_ranks if r in self.ranks]
        shaped = (isinstance(x_batches, torch.Tensor) and isinstance(y_batches, torch.Tensor) and x_batches.dim() == 3
                  and tuple(x_batches.shape[1:]) == (B, D) and tuple(y_batches.shape[1:]) == (B, C)
                  and y_batches.shape[0] == x_batches.shape[0] and x_batches.shape[0] > 0)
        nb = int(x_batches.shape[0]) if shaped else 0
        ok = (shaped and len(local_workers) == 1 and steps > 0 and self._is_pinned_f32(x_batches) and self._is_pinned_f32(y_batches)
              and os.environ.get("DTF_NATIVE_LOOP", "1") == "1")
        losses = np.zeros(max(steps, 0), np.float32)
        i = 0
        if ok:
            # the first steps of a process build the plans eagerly (both buffer parities) and graph them
            plans = self._plans()
            while i < steps and not plans.get("graphed"):
                b = (first + i * stride) % nb
                losses[i] = self.step(x_batches[b], y_batches[b], sync_loss=True)
                i += 1
                if plans["runs"] >= 4 and not plans.get("graphed"):
                    ok = False                     # graphing is switched off (DTF_E2E_GRAPH=0): stay on step()
                    break
        if not ok:
            while i < steps:
                b = (first + i * stride) % max(nb, 1)
                if local_workers and nb:
                    out = self.step(x_batches[b], y_batches[b], sync_loss=True)
                    losses[i] = out if out is not None else 0.0
                elif local_workers:
                    raise ValueError("train_loop needs pinned fp32 host batches [nb, %d, %d] / [nb, %d, %d]" % (B, D, B, C))
                else:
                    self.step(sync_loss=False)
                i += 1
            return losses
        if i == steps:
            return losses
        r = local_workers[0]
        rk, d = self.ranks[r], self._w[r]
        for old in list(plans["pending"].values()):      # deferred read-backs of step(): let them land first
            old.result()
        plans["pending"].clear()
        n = steps - i
        st = plans.get("loop_state")
        if st is None or st["rows"] < n:
            rows = max(n, 256)
            host = torch.zeros(rows, 16, dtype=torch.float32)
            if torch.cuda.is_available():
                host = host.pin_memory()
            st = plans["loop_state"] = {"rows": rows, "host": host, "np": host.numpy(), "args": LoopArgs()}
        a = st["args"]
        cp, cm = plans["copy"][r], plans["compute"][r]
        a.device, a.steps, a.depth, a.parity = rk.device.index, n, max(1, min(int(depth), 64)), plans["parity"]
        b0 = (first + i * stride) % nb
        a.prefetched = int(plans["prefetched"] == (x_batches[b0].data_ptr(), y_batches[b0].data_ptr(), plans["parity"]))
        a.x_op, a.y_op, a.prefetch_next = 1, 2, int(bool(prefetch_next))
        for p_ in range(2):
            a.n_copy[p_], a.n_compute[p_] = cp[p_].n, cm[p_].n
            a.copy_ops[p_], a.compute_ops[p_] = ctypes.addressof(cp[p_].ops), ctypes.addressof(cm[p_].ops)
        psp = plans["ps"].get(r)
        a.n_ps, a.ps_ops, a.ps_stream = (psp.n, ctypes.addressof(psp.ops), psp.stream) if psp is not None else (0, None, None)
        a.copy_stream, a.stream = cp[0].stream, cm[0].stream
        a.x_base, a.y_base = x_batches.data_ptr(), y_batches.data_ptr()
        a.x_stride, a.y_stride = B * D * 4, B * C * 4
        a.nbatches, a.first, a.batch_step = nb, b0, stride % nb
        a.loss_src, a.loss_bytes = d["loss_ptr"], self.head_ctas * 4
        a.loss_host, a.loss_row_bytes = st["host"].data_ptr(), 64
        rc = self.lib.dtf_run_loop(ctypes.byref(a))
        if rc:
            raise RuntimeError("native training loop failed with code %d (op %d of a plan, code %d)" % (rc, rc // 100000 - 1, rc % 100000))
        cuda_lib._bump(int(a.kernels))
        plans["parity"], plans["prefetched"] = int(a.parity), None
        if a.prefetched:
            bn = (first + steps * stride) % nb
            plans["prefetched"] = (x_batches[bn].data_ptr(), y_batches[bn].data_ptr(), int(a.parity))
        plans["runs"] += n
        rk.step += n
        losses[i:] = st["np"][:n, :self.head_ctas].sum(axis=1)
        return losses

    def enqueue_local_steps(self, n: int = 1, source: str = "dataset") -> int:
        """Enqueue ``n`` steps for every local rank (no host sync).  Returns the kernels launched."""
        before = cuda_lib.launch_count()
        for _ in range(n):
            self.step(sync_loss=False, source=source)
        return cuda_lib.launch_count() - before

    def capture_graphs(self, unroll: int = 16, source: str = "dataset") -> Dict[int, Any]:
        """Capture ``unroll`` steps of every local rank's stream into a CUDA graph (launch-bound inner loop).
        Everything step-dependent (wait targets, batch index) is read from device counters, so a graph can be
        replayed any number of times.  Call after at least one eager step (first-launch attribute setup)."""
        if not self.tf32 and self.cfg.sync and self.R < self.cfg.num_workers:
            raise NotImplementedError("bf16 engine with backup workers (replicas_to_aggregate < replicas): the consumed-push wait "
                                      "takes a host-side step number -- run eagerly, or use precision='tf32'")
        graphs: Dict[int, Any] = {}
        self.synchronize()
        for r, rk in self.ranks.items():
            with torch.cuda.device(rk.device):
                g = torch.cuda.CUDAGraph()
                before = cuda_lib.launch_count()
                with torch.cuda.graph(g, stream=rk.stream, capture_error_mode="thread_local"):
                    if rk.ps_stream is not None:             # fork: the shard's applies form a parallel branch of the graph
                        fork = torch.cuda.Event()
                        fork.record(rk.stream)
                        rk.ps_stream.wait_event(fork)
                    for _ in range(unroll):
                        if r in self.worker_ranks:
                            self.enqueue_worker_step(r, source)
                        if r in self.ps_ranks:
                            for _k in range(1 if self.cfg.sync else self.cfg.num_workers):
                                self.enqueue_ps_apply(r)
                    if rk.ps_stream is not None:             # join
                        join = torch.cuda.Event()
                        join.record(rk.ps_stream)
                        rk.stream.wait_event(join)
                graphs[r] = (g, cuda_lib.launch_count() - before)
                cuda_lib._bump(-(cuda_lib.launch_count() - before))      # capture launched nothing
        self._graphs = graphs
        self._graph_unroll = unroll
        return graphs

    def replay_graphs(self, times: int = 1) -> int:
        """Replay the captured graphs ``times`` times on every local rank; returns kernels launched."""
        n = 0
        for _ in range(times):
            for r, (g, k) in self._graphs.items():
                rk = self.ranks[r]
                with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
                    g.replay()
                n += k
        cuda_lib._bump(n)
        return n

    # ------------------------------------------------------------------------------------------------
    # forward only: validation / prediction on the fabric (reference distributed_mnist.py:160-165, distributed_mnist_predict.py:28-43)
    # ------------------------------------------------------------------------------------------------
    def evaluate(self, x, y=None, rank: Optional[int] = None) -> Dict[str, Any]:
        """Forward pass of the CURRENT parameters over ``x`` ([N, in_dim], any N; host or device fp32) on a local worker GPU,
        enqueued behind that worker's training steps: returns ``{"logits": [N, classes] (device), "loss": batch-SUM clipped
        cross-entropy (if ``y`` one-hot [N, classes] is given), "accuracy", "correct"}``.  Nothing is pushed, no token is
        consumed, the step counter does not move.  tf32 engines run the step kernel in forward-only mode over 128-row
        tiles (TMA-fed TF32 MMAs, parameters read from the worker's replica / the ps); bf16 engines run the bf16 GEMM +
        softmax kernels of the op layer on the ps's published parameters."""
        r = rank if rank is not None else next(q for q in self.worker_ranks if q in self.ranks)
        rk, d = self.ranks[r], self._w[r]
        spec = self.spec
        C, D = spec.classes, spec.in_dim
        with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
            xd = torch.as_tensor(x, dtype=torch.float32).to(rk.device, non_blocking=True).contiguous()
            N = xd.shape[0]
            yd = None if y is None else torch.as_tensor(y, dtype=torch.float32).to(rk.device, non_blocking=True).contiguous()
            lab = yd if yd is not None else torch.zeros((N, C), dtype=torch.float32, device=rk.device)
            logits = torch.empty((N, C), dtype=torch.float32, device=rk.device)
            if self.tf32:
                ch = min(128, 16 * self.step_ctas)        # phase 2 finalises <= 16 rows per CTA
                nch = (N + ch - 1) // ch
                lossbuf = torch.zeros((nch, 16), dtype=torch.float32, device=rk.device)
                for i in range(nch):
                    rows = min(ch, N - i * ch)
                    a = self._step_args(d, xd.data_ptr() + i * ch * D * 4, rows, lab.data_ptr() + i * ch * C * 4, 0, rows)
                    a.forward_only, a.num_signals = 1, 0
                    a.logits_out, a.loss_out = logits.data_ptr() + i * ch * C * 4, lossbuf.data_ptr() + i * 64
                    rc = self.lib.dtf_mlp_step(ctypes.byref(a), rk.stream.cuda_stream)
                    assert rc == 0, "mlp_step(forward_only) rc=%d" % rc
                cuda_lib._bump(nch)
                loss = lossbuf.sum() if yd is not None else None
            else:
                lay = self.layout
                if rk.rank in self.ps_ranks or self.world == 1:
                    pv = {k: self._var_view(rk, "master", lay[k]) for k in ("hid_w", "hid_b", "sm_w", "sm_b")}
                else:
                    pv = {k: self._peer_var_view(r, lay[k]) for k in ("hid_w", "hid_b", "sm_w", "sm_b")}
                # wait for the apply that follows this worker's last step (same acquire the next training step would do)
                for s_ in range(self.cfg.num_ps):
                    rc = self.lib.dtf_wait_token(rk.bufs["mailbox_w%d" % self.worker_ranks.index(r)].ptr + s_ * self.mb_bytes, 0,
                                                 d["stepctr_ptr"], self.cfg.timeout_ns, d["err_ptr"], rk.stream.cuda_stream)
                    assert rc == 0, rc
                h = cuda_lib.gemm(xd, pv["hid_w"].contiguous(), bias=pv["hid_b"].contiguous(), relu=True, precision="bf16")
                logits = cuda_lib.gemm(h, pv["sm_w"].contiguous(), bias=pv["sm_b"].contiguous(), precision="bf16")
                loss = None
                if yd is not None:
                    loss, _ = cuda_lib.softmax_xent_fwd_bwd(logits, yd, self.cfg.clip_min, reduce_sum=True)
            out: Dict[str, Any] = {"logits": logits}
            if yd is not None:
                pred = cuda_lib.argmax_rows(logits)
                correct = int((pred == yd.argmax(dim=1)).sum())
                out.update(loss=float(loss), correct=correct, accuracy=correct / max(N, 1), count=N)
        # the returned device tensors were produced on the worker's stream: whatever stream the caller works on waits for it
        torch.cuda.current_stream(rk.device).wait_stream(rk.stream)
        return out

    def predict(self, x, rank: Optional[int] = None) -> torch.Tensor:
        """argmax of the forward pass (reference distributed_mnist_predict.py:33,41) as an int64 device tensor."""
        r = rank if rank is not None else next(q for q in self.worker_ranks if q in self.ranks)
        rk = self.ranks[r]
        logits = self.evaluate(x, None, rank=r)["logits"]
        with torch.cuda.device(rk.device), torch.cuda.stream(rk.stream):
            pred = cuda_lib.argmax_rows(logits)
        torch.cuda.current_stream(rk.device).wait_stream(rk.stream)
        return pred

    def _peer_var_view(self, r: int, lay: VarLayout) -> torch.Tensor:
        buf = self.peer[(r, "master%d" % lay.shard)]
        return buf.tensor(torch.float32, lay.offset * 4, lay.numel_padded).view(lay.rows, lay.pitch)[:, :lay.cols]

    def read_loss(self, rank: Optional[int] = None) -> Optional[float]:
        for r in ([rank] if rank is not None else self.worker_ranks):
            if r in self.ranks:
                rk = self.ranks[r]
                w = self.worker_ranks.index(r)
                rk.stream.synchronize()
                # misc[0 : head_ctas] hold the per-CTA partials of the batch-sum loss
                return float(rk.bufs["misc_w%d" % w].tensor(torch.float32, 0, self.head_ctas).cpu().sum())
        return None

    def check_errors(self) -> None:
        for r, rk in self.ranks.items():
            rk.sync()
            if r in self.worker_ranks:
                w = self.worker_ranks.index(r)
                e = int(rk.bufs["misc_w%d" % w].tensor(torch.int32, 72, 1).cpu()[0])
                if e:
                    raise RuntimeError("worker %d: device-side wait timed out (code %d)" % (w, e))
            if r in self.ps_ranks:
                s = self.ps_ranks.index(r)
                e = int(rk.bufs["ctl%d" % s].tensor(torch.int32, self.off["err"], 1).cpu()[0])
                if e:
                    raise RuntimeError("ps shard %d: device-side wait timed out (code %d)" % (s, e))

    def synchronize(self) -> None:
        for rk in self.ranks.values():
            rk.sync()

    def join_streams(self) -> None:
        """Make every local worker stream wait for the work enqueued so far on its GPU's ps stream (so that an event
        recorded next on the worker stream covers both)."""
        for rk in self.ranks.values():
            if rk.ps_stream is not None:
                rk.stream.wait_stream(rk.ps_stream)

    def close(self) -> None:
        self.synchronize()
        self.fabric.close()


def smoke_step() -> Dict[str, Any]:
    """One tiny forward+backward+apply of the flagship model on cuda:0 (ps and worker colocated)."""
    torch.cuda.set_device(0)
    fabric = Fabric(1, {0: 0})
    eng = PSTrainEngine(MLPSpec(), EngineConfig(colocated=True, optimizer={"kind": "adam", "lr": 0.01}), fabric)
    eng.init_params()
    from ..utils.mnist_data import synthetic_mnist
    xs, ys = synthetic_mnist(400, seed=7)
    losses = []
    for i in range(4):
        x = torch.from_numpy(xs[i * 100:(i + 1) * 100]).pin_memory()
        y = torch.from_numpy(ys[i * 100:(i + 1) * 100]).pin_memory()
        losses.append(eng.step(x, y))
    eng.check_errors()
    gs = eng.read_ctl(0, "global_step")
    eng.close()
    assert gs == 4, gs
    assert all(np.isfinite(losses)), losses
    return {"losses": [round(l, 3) for l in losses], "global_step": gs, "launches": cuda_lib.launch_count()}
