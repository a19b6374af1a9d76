"""Worker runtime: the process the node agent launches for every replica of a benchmark job.

Reads the environment contract injected by the controller (the reference's 13 variables,
/root/reference/pkg/controller/pod.go:548-652, plus the torch / elastic dialect added in
``controller/pod.py``), joins ``torch.distributed`` (NCCL over NVLink 5 / NVSwitch on GPUs, gloo on
CPU), builds the requested model and runs the measured training loop:

* every step: H2D of the step's inputs from pinned memory, forward, backward + bucketed all-reduce,
  fused optimizer sweep, D2H of the loss;
* timing: W untimed warm-up steps, then exactly K steps bracketed by barrier + synchronize, CUDA
  events on the device, max over ranks; rank 0 writes the result JSON and patches it onto the job;
* elastic (``runtime.elastic``): a side thread watches ``status.rendezvous``; at a step boundary all
  ranks agree on the newest generation, tear the process group down and re-rendezvous with the new
  world size; survivors keep params / optimizer state / step on the device and broadcast them to
  joiners; ranks that fall out of range leave with exit 0;
* restart: ``TRAININGJOB_REPLICA_RESTARTCOUNT`` > 0 => resume from the newest checkpoint written (asynchronously,
  ``runtime.checkpoint``) by rank 0 every ``--ckpt-every`` steps (SURVEY.md §5.4);
* ``faultTolerant`` elastic jobs: a collective that fails because a peer died does not end the process -- the step is
  discarded, the group dropped, and the loop continues on the controller's next generation (``runtime.rendezvous``).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import signal
import sys
import time
from typing import Any, Dict, List, Optional

import torch
import torch.distributed as dist

from .elastic import ElasticWatcher, env_int, rendezvous_from_env
from .rendezvous import (StaleGeneration, StallBreaker, heartbeat, init_process_group, max_over_ranks,  # noqa: F401
                         rendezvous, sync_state, teardown_group, wait_for_newer_generation)
from .trainer import EngineTrainer, SyntheticTokens


# ------------------------------------------------------------------------------------ adapters
class EngineAdapter:
    """GPT-2 / BERT-shaped transformer on the hand-written engine (CUDA only)."""

    def __init__(self, name: str, batch: int, seq: int, args, device: str = "cuda"):
        """``device``: always "cuda" in a worker (``build_adapter``); the CPU dry-run tests pass "cpu" together with
        emulated kernel entry points (tests/kernel_emulation.py) to execute the adapter's control flow."""
        from ..models.gpt2 import GPT2Config, GPT2Engine, flops_per_token

        if name in ("bert", "bert-tiny"):
            # the real thing: word + position + token-type embeddings, post-LN bidirectional encoder, MLM head and loss
            from ..models.bert import BertConfig, BertEngine, SyntheticMLM, bert_flops_per_token

            cfg = BertConfig.base() if name == "bert" else BertConfig.tiny()
            seq = min(seq, cfg.block_size)
            self.engine = BertEngine(cfg, batch, seq, device, seed=args.seed, gemm_backend=args.gemm)
            self.data = SyntheticMLM(cfg.vocab_size, batch, seq, n_batches=4, seed=args.seed + 1, pin=device != "cpu")
            self.flops_per_step = bert_flops_per_token(cfg, seq) * batch * seq
        else:
            if name == "gpt2":
                cfg = GPT2Config.small()
            elif name == "gpt2-tiny":
                cfg = GPT2Config.tiny()
            else:
                raise ValueError(name)
            seq = min(seq, cfg.block_size)
            self.engine = GPT2Engine(cfg, batch, seq, device, seed=args.seed, gemm_backend=args.gemm, causal=True)
            self.data = SyntheticTokens(cfg.vocab_size, batch, seq, n_batches=4, seed=args.seed + 1)
            self.flops_per_step = flops_per_token(cfg, seq) * batch * seq
        self.cfg = cfg
        self.batch, self.seq = batch, seq
        self.h2d_bytes = self.data.bytes_per_step
        self.d2h_bytes = 4
        self.trainer: Optional[EngineTrainer] = None
        self.args = args
        self.describe = {"model": cfg.name, "seq_len": seq, "params": self.engine.num_parameters(),
                         "gemm": args.gemm}

    def bind(self, group=None) -> None:
        old = self.trainer
        # a faultTolerant job survives the loss of a peer in place, which needs every rank to hold the whole optimizer
        # state and a collective that can be aborted: library all-reduce instead of the owner-sharded peer-memory path
        allreduce = "nccl" if os.environ.get("AITJ_FAULT_TOLERANT") == "1" and "AITJ_ALLREDUCE" not in os.environ else None
        self.trainer = EngineTrainer(self.engine, lr=self.args.lr, use_graph=not self.args.no_graph, group=group,
                                     allreduce=allreduce)
        if old is not None:
            self.trainer.step_count = old.step_count

    def train_step(self) -> float:
        return self.trainer.step(*self.data.next())

    def discard_step(self) -> None:
        self.engine.params.g32.zero_()
        if self.engine.params.g_small is not None:
            self.engine.params.g_small.zero_()

    def prepare_state(self) -> None:
        """Collective.  With the owner-sharded optimizer every rank only keeps its own range of the fp32 master weights
        and moments current: gather them so that ``state_tensors`` is the whole state on every rank (before a
        checkpoint, before the process group is re-formed)."""
        sh = self.engine.params.shard
        if sh is None or not dist.is_initialized():
            return
        P = self.engine.params
        for r in range(sh.world):
            a, b = sh.bounds[r], sh.bounds[r + 1]
            if b > a:
                for t in (P.p32, P.m, P.v):
                    dist.broadcast(t[a:b], src=r)

    def state_tensors(self) -> List[torch.Tensor]:
        return self.engine.params.state_tensors()

    def after_state_load(self) -> None:
        self.engine.params.refresh_compute_copy()

    @property
    def step_count(self) -> int:
        return self.trainer.step_count if self.trainer else 0

    @step_count.setter
    def step_count(self, v: int) -> None:
        if self.trainer:
            self.trainer.step_count = v

    def launches_per_step(self) -> int:
        t = self.trainer
        if t.launches_per_step:
            return t.launches_per_step
        return 0


class TorchAdapter:
    """nn.Module models (MNIST CNN, ResNet-50, CPU MLP) through ``parallel.flat_ddp``."""

    def __init__(self, name: str, batch: int, args, device: torch.device):
        from ..models.mnist_cnn import MLP, MnistCNN

        self.name, self.batch, self.dev, self.args = name, batch, device, args
        g = torch.Generator().manual_seed(args.seed + 1)
        torch.manual_seed(args.seed)       # the modules below draw their initial weights from the global generator
        if name == "mnist":
            self.module = MnistCNN()
            shape, ncls = (1, 28, 28), 10
        elif name == "resnet50":
            from ..models.resnet50 import build_resnet50

            self.module = build_resnet50()
            shape, ncls = (3, 224, 224), 1000
        elif name == "mlp":
            self.module = MLP()
            shape, ncls = (64,), 10
        else:
            raise ValueError(name)
        self.module = self.module.to(device)
        self.channels_last = device.type == "cuda" and len(shape) == 3
        if self.channels_last:
            self.module = self.module.to(memory_format=torch.channels_last)
        pin = device.type == "cuda"
        self.batches = []
        for _ in range(4):
            x = torch.randn(batch, *shape, generator=g)
            y = torch.randint(0, ncls, (batch,), generator=g)
            if pin:
                x, y = x.pin_memory(), y.pin_memory()
            self.batches.append((x, y))
        self.i = 0
        self.x_dev = torch.empty(batch, *shape, device=device)
        if self.channels_last:
            self.x_dev = self.x_dev.contiguous(memory_format=torch.channels_last)
        self.y_dev = torch.empty(batch, dtype=torch.int64, device=device)
        self.h2d_bytes = self.batches[0][0].numel() * 4 + batch * 8
        self.d2h_bytes = 4
        self.ddp = None
        self._steps = 0
        self.loss_host = torch.zeros(1).pin_memory() if pin else torch.zeros(1)
        self.describe = {"model": name, "params": sum(p.numel() for p in self.module.parameters())}
        self.flops_per_step = 0.0

    def bind(self, group=None) -> None:
        from ..parallel.flat_ddp import FlatDDP

        backend = "nccl" if self.dev.type == "cuda" else "gloo"
        # CUDA: forward + backward are replayed as one CUDA graph (the step of the small networks is launch bound: MNIST
        # CNN 1.4 ms of mostly gaps), the flat gradient buffer is reduced by one collective after it
        self.use_graph = self.dev.type == "cuda" and not self.args.no_graph
        if self.ddp is None:
            self.ddp = FlatDDP(self.module, group=group, backend=backend, lr=self.args.lr,
                               optimizer="adamw" if self.name != "mlp" else "sgd", overlap=not self.use_graph)
        else:  # re-bind after a re-rendezvous: keep buffers, rebuild the reducer for the new group
            from ..parallel.ddp import BucketAllReducer

            self.ddp.group = group
            self.ddp.world = dist.get_world_size(group) if dist.is_initialized() else 1
            self.ddp.reducer = BucketAllReducer(self.ddp.g32, self.ddp.buckets, group, backend, 0) \
                if self.ddp.world > 1 else None
            if self.ddp.reducer is not None and self.ddp.overlap and not getattr(self.ddp, "_hooked", False):
                for idx, p in enumerate(self.ddp.params):
                    p.register_post_accumulate_grad_hook(self.ddp._make_hook(idx))
        self.ddp._hooked = self.ddp.reducer is not None or getattr(self.ddp, "_hooked", False)

    def _fwd_bwd(self) -> torch.Tensor:
        if self.dev.type == "cuda":
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss = torch.nn.functional.cross_entropy(self.module(self.x_dev), self.y_dev)
        else:
            loss = torch.nn.functional.cross_entropy(self.module(self.x_dev), self.y_dev)
        loss.backward()
        return loss

    def _capture(self) -> None:
        """Forward + backward of the fixed-shape step as one CUDA graph: static inputs (x_dev / y_dev), gradients
        accumulated in place into the flat buffer the parameters' ``.grad`` already point into."""
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                self._fwd_bwd()
                self.ddp.g32.zero_()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(g):
                self._graph_loss = self._fwd_bwd().detach()
            self.ddp.g32.zero_()
            self.graph = g
        except Exception as e:  # noqa: BLE001 - eager fallback (and the per-bucket overlap is gone: one all-reduce)
            self.graph_error = f"{type(e).__name__}: {e}"
            self.graph = None
            self.use_graph = False
            torch.cuda.synchronize()

    def train_step(self) -> float:
        x, y = self.batches[self.i % len(self.batches)]
        self.i += 1
        self.x_dev.copy_(x, non_blocking=True)
        self.y_dev.copy_(y, non_blocking=True)
        if getattr(self, "use_graph", False) and getattr(self, "graph", None) is None and \
                getattr(self, "graph_error", None) is None:
            self._capture()
        if getattr(self, "graph", None) is not None:
            self.graph.replay()
            loss = self._graph_loss
        else:
            loss = self._fwd_bwd()
        self.ddp.finish_backward()
        self.ddp.step()
        self._steps += 1
        self.loss_host.copy_(loss.detach().float().reshape(1), non_blocking=True)
        if self.dev.type == "cuda":
            torch.cuda.current_stream().synchronize()
        return float(self.loss_host[0])

    def discard_step(self) -> None:
        if self.ddp is not None:
            self.ddp.discard_step()        # .grad are views of the flat buffer it zeroes

    def prepare_state(self) -> None:
        return                             # every rank holds the whole state

    def state_tensors(self) -> List[torch.Tensor]:
        return self.ddp.state_tensors()

    def after_state_load(self) -> None:
        return

    @property
    def step_count(self) -> int:
        return self._steps

    @step_count.setter
    def step_count(self, v: int) -> None:
        self._steps = v
        if self.ddp is not None:
            self.ddp.step_count = v

    def launches_per_step(self) -> int:
        return 1 if self.dev.type == "cuda" else 0


def build_adapter(args, device: torch.device):
    if args.model in ("gpt2", "gpt2-tiny", "bert", "bert-tiny"):
        if device.type != "cuda":
            raise RuntimeError(f"model {args.model} needs a CUDA device (hand-written sm_100a kernels)")
        return EngineAdapter(args.model, args.batch, args.seq, args)
    return TorchAdapter(args.model, args.batch, args, device)


# ------------------------------------------------------------------------------------ checkpoint
def ckpt_path(args) -> str:
    d = args.ckpt_dir or os.path.join(os.environ.get("AITJ_WORKDIR", "/tmp"), "ckpt")
    os.makedirs(d, exist_ok=True)
    job = os.environ.get("TRAININGJOB_NAME", "job")
    # per job *object*, not per name: a job submitted again under the same name must never resume from its predecessor's
    # state (the uid survives every restart of the job's replicas, which is what a checkpoint is for)
    uid = os.environ.get("AITJ_JOB_UID", "")[:8]
    return os.path.join(d, f"{job}-{uid}.pt" if uid else f"{job}.pt")


_CKPT: Dict[str, Any] = {}


def checkpointer(args):
    """The process-wide asynchronous checkpoint writer (``runtime/checkpoint.py``)."""
    from .checkpoint import AsyncCheckpointer

    path = ckpt_path(args)
    if _CKPT.get("path") != path:
        _CKPT["path"], _CKPT["writer"] = path, AsyncCheckpointer(path)
    return _CKPT["writer"]


def save_checkpoint(args, adapter, step: int) -> None:
    """Snapshot the state in stream order and write it in the background; ``AITJ_CKPT_ASYNC=0`` waits for the file."""
    w = checkpointer(args)
    w.save(step, adapter.state_tensors())
    if os.environ.get("AITJ_CKPT_ASYNC", "1") == "0":
        w.wait()


def load_checkpoint(args, adapter) -> int:
    from .checkpoint import load_into

    if _CKPT.get("writer") is not None:
        _CKPT["writer"].wait()              # our own write in flight (in-place recovery falls back to it)
    meta = load_into(ckpt_path(args), adapter.state_tensors())
    if meta is None:
        return 0
    adapter.after_state_load()
    return int(meta["step"])


def guarded(breaker, generation: int, fn):
    """Run a collective-bearing ``fn`` as "inside a step" for the stall breaker: only a generation newer than
    ``generation`` (= another peer was lost meanwhile) makes it abort the communicator; the abort surfaces as a
    RuntimeError, which the training loop's recovery path handles."""
    if breaker is None:
        return fn()
    breaker.progress(generation)
    breaker.in_step = True
    try:
        out = fn()
    finally:
        breaker.in_step = False
    if breaker.tripped:
        raise RuntimeError("the communicator was aborted while the state hand-off was in flight")
    return out


# ------------------------------------------------------------------------------------ outputs
DUMP_SAMPLE = 1 << 22      # elements kept per state tensor: 3 x 16 MB for GPT-2 small's parameters and AdamW moments


def dump_outputs(out_dir: str, loss: float, state: List[torch.Tensor]) -> None:
    """What the last training step produced, as ``out_dir/<name>.npy`` (float32): its loss and the trained state (fp32
    parameters, then the optimizer's moments).  A tensor larger than ``DUMP_SAMPLE`` elements is cut to a fixed sample
    (sorted indices from a generator seeded with 0), so that runs of two builds on the same inputs compare element for
    element."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float32))
    for name, t in zip(("params", "exp_avg", "exp_avg_sq"), state):
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0))
            t = t.index_select(0, idx.sort().values.to(t.device))
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------ main loop
def run(args) -> Dict[str, Any]:
    t_proc = time.time()
    rank = env_int("RANK", env_int("TRAININGJOB_REPLICA_INDEX", 0))
    rdv = rendezvous_from_env()
    world, port, generation = rdv["world"], rdv["port"], rdv["generation"]
    use_cuda = torch.cuda.is_available() and not args.cpu
    device = torch.device("cuda", env_int("LOCAL_RANK", 0) if torch.cuda.device_count() > 1 else 0) \
        if use_cuda else torch.device("cpu")
    if use_cuda:
        torch.cuda.set_device(device)
    if args.elastic and os.environ.get("AITJ_FAULT_TOLERANT") == "1":
        # NCCL's watchdog would take the process down on an asynchronous communicator error or a collective timeout
        # (TearDown / SkipCleanUp); a faultTolerant job handles the loss of a peer itself (StallBreaker + recovery below)
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        # A communicator that must be abortable with a peer already dead should not hold NVSwitch multicast (NVLS)
        # objects: their teardown involves every member.  Precaution, not a measured fix -- in-place recovery is verified
        # on 2 GPUs (where NCCL does not use NVLS); the 4-GPU attempts of round 2 ended without a diagnosis
        # (profiles/r2_fault_recovery_gpu.md).  Costs the faultTolerant job's all-reduce the in-switch reduction.
        os.environ.setdefault("NCCL_NVLS_ENABLE", "0")
    trace = {"process_start": t_proc, "torch_imported": time.time()}
    heartbeat(force=True)
    watcher = ElasticWatcher.from_env(generation)
    if watcher is not None and not args.elastic:
        watcher.poll = 5.0  # reporting only
    adapter = build_adapter(args, device)
    trace["model_built"] = time.time()
    heartbeat(force=True)
    joiner = bool(args.elastic and watcher is not None and generation > 1 and world > 1)
    if joiner:
        # Joining a running job: do everything that needs no peer first -- CUDA context, model build, two throw-away
        # steps (kernel loading, cuDNN plans, allocator growth; the state is overwritten by rank 0's broadcast
        # anyway) -- and only then tell the survivors, who keep training until this rank is ready to rendezvous.
        adapter.bind(None)
        for _ in range(2):
            adapter.train_step()
        if use_cuda:
            torch.cuda.synchronize()
        trace["prewarmed"] = time.time()
        watcher.announce_ready(rank, generation)
        print(f"[worker {rank}] joiner ready for generation {generation} after "
              f"{trace['prewarmed'] - t_proc:.2f}s of local set-up (model build "
              f"{trace['model_built'] - t_proc:.2f}s, warm-up steps {trace['prewarmed'] - trace['model_built']:.2f}s)",
              flush=True)
    if world > 1:
        got = rendezvous(rank, {"generation": generation, "world": world, "port": port}, device, watcher)
        if got is None:
            print(f"[worker {rank}] not part of the current world any more, leaving", flush=True)
            return {"left": True, "generation": generation, "step": 0}
        generation, world, port = got["generation"], got["world"], got["port"]
        if watcher is not None:
            watcher.adopted(generation, world)
    trace["rendezvous_done"] = time.time()
    heartbeat(force=True)
    adapter.bind(None)
    print(f"[worker {rank}] world {world}: gradient sync = "
          f"{getattr(getattr(adapter, 'trainer', None), 'allreduce_backend', 'flat buffer all-reduce (nccl / gloo)')}",
          flush=True)

    restart_count = env_int("TRAININGJOB_REPLICA_RESTARTCOUNT", 0)
    start_step = 0
    if restart_count > 0 and args.ckpt_every > 0:
        start_step = load_checkpoint(args, adapter)
        adapter.step_count = start_step
        print(f"[worker {rank}] restart #{restart_count}: resumed from checkpoint at step {start_step}", flush=True)
    # a joiner without a checkpoint only has its throw-away warm-up state: it must never be elected as the source
    joined_step = sync_state(adapter, start_step, device, have_state=not joiner or start_step > 0)
    if joiner:
        print(f"[worker {rank}] joined generation {generation} (world {world}) at step {joined_step}", flush=True)
    # faultTolerant (types.go:47, never read by the reference): the loss of a peer is survived in place -- see the
    # except branch of the training loop
    fault_tolerant = bool(args.elastic and watcher is not None and os.environ.get("AITJ_FAULT_TOLERANT") == "1")
    breaker = None
    # (armed on CUDA, where a collective with a dead peer hangs instead of raising; AITJ_STALL_BREAKER=force arms it for
    #  any backend -- the CPU tests use it with collectives that are made to hang the way NCCL's do)
    hangs = use_cuda or os.environ.get("AITJ_STALL_BREAKER") == "force"
    if fault_tolerant and hangs and float(os.environ.get("AITJ_FT_ABORT_AFTER", "3")) > 0:
        breaker = StallBreaker(watcher, float(os.environ.get("AITJ_FT_ABORT_AFTER", "3")))
    elif watcher is not None and hangs and world > 1 and float(os.environ.get("AITJ_STALL_EXIT_AFTER", "3")) > 0:
        # not faultTolerant: a rank stuck behind a dead peer cannot be repaired in place; once the controller has started
        # to repair the job (newer generation) it leaves at once instead of waiting for the heartbeat time-out
        breaker = StallBreaker(watcher, float(os.environ.get("AITJ_STALL_EXIT_AFTER", "3")), action="exit")
    recoveries: List[Dict[str, Any]] = []

    stop = {"flag": False}
    signal.signal(signal.SIGTERM, lambda *_: stop.__setitem__("flag", True))

    total = args.warmup + args.steps if args.steps > 0 else 1 << 60
    losses: List[float] = []
    rescales: List[Dict[str, Any]] = []
    timing: Dict[str, Any] = {}
    ev0 = ev1 = None
    t_wall0 = 0.0
    t_epoch0 = 0.0
    timed_from = -1          # first step inside the timed region (-1: not armed yet)
    step = joined_step
    first_step_done = False
    warmed_generation = -1          # generation whose trainer has completed at least one step
    pending_rescale = None
    from ..ops import lib as oplib

    launches0 = 0
    # rank 0 publishes its wall-clock throughput every AITJ_REPORT_EVERY seconds (0 = only the final, device-timed result)
    report_every = float(os.environ.get("AITJ_REPORT_EVERY", "10"))
    live_t0, live_step0 = time.time(), step
    while step < total and not stop["flag"]:
        if breaker is not None:
            breaker.progress(generation)
            # the first step on a freshly bound trainer captures CUDA graphs / loads kernels: seconds, not a stall
            breaker.patience = breaker.after_s if warmed_generation == generation else max(breaker.after_s, 30.0)
        failure = None
        try:
            # ---- elastic: agree on the newest rendezvous generation at the step boundary ------------
            if watcher is not None and args.elastic:
                target = watcher.agree(device, guard=breaker)
                if target is not None and target["generation"] != generation:
                    t0 = time.time()
                    new_world = target["world"]
                    print(f"[worker {rank}] rendezvous generation {generation} -> {target['generation']} "
                          f"(world {world} -> {new_world}) at step {step}", flush=True)
                    if dist.is_initialized():
                        adapter.prepare_state()       # sharded optimizer state -> whole state on every survivor
                        if use_cuda:
                            torch.cuda.synchronize()
                        dist.destroy_process_group()
                    if rank >= new_world:
                        print(f"[worker {rank}] leaving: world shrinks to {new_world} (generation {target['generation']})",
                              flush=True)
                        return {"left": True, "generation": target["generation"], "step": step}
                    generation, world, port = target["generation"], new_world, target["port"]
                    t1 = time.time()
                    if world > 1:
                        got = rendezvous(rank, {"generation": generation, "world": world, "port": port}, device, watcher)
                        if got is None:
                            return {"left": True, "generation": generation, "step": step}
                        generation, world, port = got["generation"], got["world"], got["port"]
                    t2 = time.time()
                    adapter.bind(None)
                    step = guarded(breaker, generation, lambda: sync_state(adapter, step, device))
                    heartbeat(force=True)
                    watcher.adopted(generation, world)
                    pending_rescale = {"generation": generation, "world": world, "t0": t0,
                                       "observed_at": target.get("observed_at", t0),
                                       "teardown_s": t1 - t0, "init_pg_s": t2 - t1, "sync_state_s": time.time() - t2}
                    continue    # back to the step boundary: every rank (joiners included) runs the same sequence
            # ---- timed region bookkeeping ----------------------------------------------------------------
            # armed at the first step boundary at or past the warm-up: a replica resumed from a checkpoint (or an
            # elastic joiner) starts past `--warmup` and still gets a timed region (and counts the steps it timed)
            if timed_from < 0 and step >= args.warmup and args.steps > 0:
                if world > 1:
                    dist.barrier()
                if use_cuda:
                    torch.cuda.synchronize()
                    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    ev0.record()
                t_wall0 = time.perf_counter()
                t_epoch0 = time.time()
                timed_from = step
                launches0 = oplib.LAUNCHES
            if breaker is not None:
                breaker.progress(generation)
                breaker.in_step = True
            try:
                loss = adapter.train_step()
            finally:
                if breaker is not None:
                    breaker.in_step = False
            warmed_generation = generation
            if breaker is not None and breaker.tripped:
                raise RuntimeError("the communicator was aborted while this step was in flight")
        except RuntimeError as e:
            # ---- faultTolerant: a peer died under a collective -----------------------------------------------------
            # (gloo raises in the survivors; for NCCL the StallBreaker aborts the communicator.)  The survivors keep
            # their process, device state and -- on GPUs -- CUDA context: drop the broken group, wait for the
            # controller to replace the lost replica (restart scope Pod, new rendezvous generation), re-rendezvous and
            # continue from the survivors' state.  Without faultTolerant the error ends this replica and the job's
            # restartPolicy / restartScope take over, as in the reference (pod.go:208-250).
            if not fault_tolerant or world <= 1:
                raise
            failure = (type(e).__name__, (str(e).splitlines() or [""])[0][:160])
        if failure is not None:
            # (outside the except block: the traceback of the failed step references the work handles of the broken
            # group, and with them its sockets)
            t0 = time.time()
            aborted = breaker is not None and breaker.tripped
            print(f"[worker {rank}] step {step}: lost a peer ({failure[0]}: {failure[1]}); "
                  f"keeping state, waiting for the next rendezvous generation", flush=True)
            # pending work handles keep the group's sockets open; a peer that is blocked on *us* (gloo does not
            # propagate a failure beyond the dead rank's direct neighbours) only errors out once they really close
            adapter.discard_step()
            teardown_group(broken=True)
            gc.collect()
            target = wait_for_newer_generation(watcher, generation, float(os.environ.get("AITJ_FT_WAIT", "120")),
                                               should_stop=lambda: stop["flag"])
            if target is None and stop["flag"]:
                print(f"[worker {rank}] terminated while waiting for the job to be repaired", flush=True)
                break
            if target is None:
                print(f"[worker {rank}] no new rendezvous generation was published: giving up", flush=True)
                raise RuntimeError(f"collective failed and the job was not repaired: {failure[0]}: {failure[1]}")
            if rank >= target["world"]:
                print(f"[worker {rank}] leaving: world shrinks to {target['world']} (generation {target['generation']})",
                      flush=True)
                return {"left": True, "generation": target["generation"], "step": step}
            t1 = time.time()
            got = rendezvous(rank, {"generation": target["generation"], "world": target["world"],
                                    "port": target["port"]}, device, watcher)
            if got is None:
                return {"left": True, "generation": target["generation"], "step": step}
            generation, world, port = got["generation"], got["world"], got["port"]
            t2 = time.time()
            if aborted and args.ckpt_every > 0 and os.path.exists(ckpt_path(args)):
                # kernels released by an abort ran on with whatever the dead peer left in the buffers: do not trust
                # this rank's copy when there is a checkpoint to fall back to
                step = load_checkpoint(args, adapter)
                adapter.step_count = step
            if breaker is not None:
                breaker.tripped = False
                breaker.progress(generation)
            adapter.bind(None)
            # the hand-off is a chain of collectives on the new group: if ANOTHER peer dies under it, a still newer
            # generation is published and the breaker must be able to get this rank out of it
            try:
                step = guarded(breaker, generation, lambda: sync_state(adapter, step, device))
            except RuntimeError as e:
                # (this block is outside the loop's try: handled here.)  The group is gone again; the step boundary's
                # generation agreement finds the newest record and joins it through the ordinary rescale path.
                print(f"[worker {rank}] another peer was lost during the state hand-off of generation {generation} "
                      f"({type(e).__name__}); joining the next generation", flush=True)
                teardown_group(broken=True)
                if breaker is not None:
                    breaker.tripped = False
                continue
            heartbeat(force=True)
            watcher.adopted(generation, world)
            pending_rescale = {"generation": generation, "world": world, "t0": t0, "observed_at": t0,
                               "teardown_s": t1 - t0, "init_pg_s": t2 - t1, "sync_state_s": time.time() - t2,
                               "recovered_from": failure[0]}
            continue
        losses.append(loss)
        step += 1
        heartbeat()
        if pending_rescale is not None:
            # the first completed step at the new world size ends the rescale
            now = time.time()
            rec = {"generation": pending_rescale["generation"], "world": pending_rescale["world"],
                   "seconds": now - pending_rescale["t0"], "since_change": now - pending_rescale["observed_at"],
                   "teardown_s": round(pending_rescale["teardown_s"], 4),
                   "init_pg_s": round(pending_rescale["init_pg_s"], 4),
                   "sync_state_s": round(pending_rescale["sync_state_s"], 4)}
            rec["first_step_s"] = round(rec["seconds"] - rec["teardown_s"] - rec["init_pg_s"] - rec["sync_state_s"], 4)
            if "recovered_from" in pending_rescale:
                rec["recovered_from"] = pending_rescale["recovered_from"]
                recoveries.append(rec)
            rescales.append(rec)
            print(f"[worker {rank}] step {step}: rescaled to world={rec['world']} gen={rec['generation']} in "
                  f"{rec['seconds']:.3f}s", flush=True)
            if watcher is not None:
                watcher.report_rescale(rank, rec, force="recovered_from" in rec)   # rank 0 may be the replaced one
            pending_rescale = None
        if not first_step_done:
            first_step_done = True
            trace["first_step_done"] = time.time()
            if watcher is not None:
                watcher.report_trace(rank, trace)
        if rank == 0 and watcher is not None and report_every > 0 and time.time() - live_t0 >= report_every:
            dt, n = time.time() - live_t0, step - live_step0
            if n > 0:
                watcher.report_live(rank, {"samples_per_sec": round(args.batch * world * n / dt, 2),
                                           "ms_per_step": round(dt * 1e3 / n, 3), "world": world, "steps_done": step,
                                           "global_batch": args.batch * world, "recoveries": len(recoveries)})
            live_t0, live_step0 = time.time(), step
        if args.ckpt_every > 0 and step % args.ckpt_every == 0:
            adapter.prepare_state()
            if rank == 0:
                save_checkpoint(args, adapter, adapter.step_count)
        if args.step_sleep > 0:
            time.sleep(args.step_sleep)

    result: Dict[str, Any] = {"rank": rank, "world": world, "steps_done": step, "generation": generation,
                              "final_loss": losses[-1] if losses else None, "rescales": rescales,
                              "recoveries": recoveries, "trace": trace}
    if breaker is not None:
        breaker.stop()
    if _CKPT.get("writer") is not None:
        _CKPT["writer"].wait(60.0)
    n_timed = step - timed_from if timed_from >= 0 else 0
    if args.steps > 0 and step >= total and n_timed > 0:
        if use_cuda:
            ev1.record()
            torch.cuda.synchronize()
        t_epoch1 = time.time()
        if world > 1:
            dist.barrier()
        wall = time.perf_counter() - t_wall0
        dev_ms = ev0.elapsed_time(ev1) if use_cuda else wall * 1e3
        dev_ms = max_over_ranks(dev_ms, device)
        global_batch = args.batch * world
        result.update({"timed_steps": n_timed, "timed_from_step": timed_from,
                       "timed_region_epoch": [t_epoch0, t_epoch1]})
        graph_launches = adapter.launches_per_step()
        eager_launches = (oplib.LAUNCHES - launches0)
        result.update({
            "ms_per_step": dev_ms / n_timed,
            "samples_per_sec": global_batch * n_timed / (dev_ms / 1e3),
            "wall_ms_per_step": wall * 1e3 / n_timed,
            "global_batch": global_batch, "batch_per_gpu": args.batch,
            "h2d_bytes_per_step": adapter.h2d_bytes, "d2h_bytes_per_step": adapter.d2h_bytes,
            "gpu_launches": graph_launches * n_timed if graph_launches else eager_launches,
            "launches_per_step": graph_launches or (eager_launches // max(1, n_timed)),
            "loss_first": losses[0] if losses else None, "loss_last": losses[-1] if losses else None,
            "flops_per_step": getattr(adapter, "flops_per_step", 0.0),
            "describe": adapter.describe,
            "cuda_graph": bool(getattr(getattr(adapter, "trainer", None), "graph", None)
                               or getattr(getattr(adapter, "trainer", None), "seg_graphs", None)
                               or getattr(adapter, "graph", None)),
            "graph_segments": len(getattr(getattr(adapter, "trainer", None), "seg_graphs", None) or []) or None,
            "graph_error": getattr(getattr(adapter, "trainer", None), "graph_error", None)
            or getattr(adapter, "graph_error", None),
            "allreduce": getattr(getattr(adapter, "trainer", None), "allreduce_backend", "nccl" if world > 1 else "none"),
        })
        if args.dump_outputs:
            adapter.prepare_state()         # collective: the whole trained state on every rank
            if rank == 0:
                dump_outputs(args.dump_outputs, losses[-1], adapter.state_tensors())
    if rank == 0 and args.result:
        os.makedirs(os.path.dirname(os.path.abspath(args.result)), exist_ok=True)
        with open(args.result + ".tmp", "w") as f:
            json.dump(result, f)
        os.replace(args.result + ".tmp", args.result)
    if rank == 0 and watcher is not None:
        watcher.report_result(result)
    if dist.is_initialized():
        try:
            dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass
    return result


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="aitj-worker")
    ap.add_argument("--model", default="gpt2", choices=["gpt2", "gpt2-tiny", "bert", "bert-tiny", "resnet50", "mnist", "mlp"])
    ap.add_argument("--batch", type=int, default=16, help="per-GPU batch size")
    ap.add_argument("--seq", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (0 = run until SIGTERM)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--gemm", default="tcgen05", choices=["tcgen05", "cublas"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--cpu", action="store_true")
    ap.add_argument("--elastic", action="store_true")
    ap.add_argument("--result", default="")
    ap.add_argument("--ckpt-dir", default="")
    ap.add_argument("--ckpt-every", type=int, default=0)
    ap.add_argument("--step-sleep", type=float, default=0.0)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the last step's loss and a sample of the trained state to DIR")
    return ap.parse_args(argv)


def main(argv=None) -> int:
    args = parse_args(argv)
    res = run(args)
    if res.get("samples_per_sec"):
        print(f"[worker {res['rank']}] {res['samples_per_sec']:.1f} samples/s  {res['ms_per_step']:.3f} ms/step "
              f"loss {res.get('loss_first')} -> {res.get('loss_last')}", flush=True)
    return 0


def _record_exit(code: int) -> None:
    """``$AITJ_EXIT_FILE``: lets an agent that adopted this process after a restart (and therefore cannot wait() for
    it) still learn how it ended."""
    path = os.environ.get("AITJ_EXIT_FILE", "")
    if not path:
        return
    try:
        with open(path, "w") as f:
            f.write(str(int(code)))
    except OSError:
        pass


def cli() -> None:
    """Process entry point (``python -m ...runtime.worker`` and the ``aitj-worker`` script): runs ``main`` and records the
    exit code in ``$AITJ_EXIT_FILE`` however it ends."""
    try:
        code = main()
    except SystemExit as e:
        code = e.code if isinstance(e.code, int) else (0 if e.code is None else 1)
        _record_exit(code)
        raise
    except BaseException:
        _record_exit(1)
        raise
    _record_exit(code)
    sys.exit(code)


if __name__ == "__main__":
    cli()
