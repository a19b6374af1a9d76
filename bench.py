#!/usr/bin/env python
"""Headline benchmark (driver contract): samples/sec of the launched DDP training job.

    python bench.py --gpus N --steps K --warmup W [--model gpt2|bert|resnet50|mnist] [--dump-outputs DIR]

* ``value``  -- device-timed (CUDA events, max over ranks) whole-job samples/sec of the flagship
  training step (GPT-2 small, seq 1024, bf16, per-GPU batch 16 = weak scaling) run by the ranks the
  driver launched (``torchrun`` for N>1): every step = H2D of the step's tokens from pinned memory,
  forward, backward + bucketed all-reduce, fused AdamW, D2H of the loss.
* ``e2e``    -- the same metric measured through the repo's public API: rank 0 brings up the local
  control plane (API server + node agent + operator), ``apply``-s an ``AITrainingJob`` with N replicas
  and reads the samples/sec its controller-launched workers report (fresh processes, one per GPU,
  pinned with CUDA_VISIBLE_DEVICES, NCCL over NVLink); also reports reconcile->running latency.
* ``--dump-outputs DIR`` -- after the timed steps, rank 0 of the device-timed run writes what its last step computed:
  ``loss.npy`` and a fixed sample of the trained fp32 parameters and AdamW moments (``params.npy``, ``exp_avg.npy``,
  ``exp_avg_sq.npy``; float32, 48 MB at most).  Inputs and initial weights are seeded, so two builds run with the same
  arguments can be compared output for output -- within a tolerance: the fp32 atomic accumulations of the kernels
  (split-K weight gradients, bias column sums, the gradient norm) repeat to round-off, not bit for bit, and AdamW
  carries that into the weights, so two runs of one build on the GPU already differ slightly.
* ``--impl reference`` -- the reference is a Go Kubernetes operator with no Python package, no GPU
  code and no cluster to run against here: prints ``{"impl": "reference", "unavailable": ...}``.

BASELINE.json publishes no numbers (``published: {}``), so ``vs_baseline`` is null.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL_DEFAULTS = {
    "gpt2": {"batch": 16, "seq": 1024, "name": "GPT-2 small (124M) DDP"},
    "bert": {"batch": 32, "seq": 512, "name": "BERT-base DDP"},
    "resnet50": {"batch": 128, "seq": 0, "name": "ResNet-50 DDP bf16"},
    "mnist": {"batch": 512, "seq": 0, "name": "MNIST CNN DDP"},
    "gpt2-tiny": {"batch": 4, "seq": 128, "name": "GPT-2 tiny (smoke)"},
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self):
        self.proc = None
        self.path = os.path.join(tempfile.gettempdir(), f"aitj_clocks_{os.getpid()}.csv")

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self, window=None):
        """``window`` = (t0, t1) epoch seconds of the timed region: only samples taken inside it are summarised (the
        process spends most of its life importing / initialising at idle clocks, which used to drown the median)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        self.f.close()
        import datetime

        sm, mx, reasons, power = [], [], set(), []
        rows = []
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            ts = None
            if len(p) >= 10:
                try:
                    ts = datetime.datetime.strptime(p[9], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    ts = None
            rows.append((ts, p))
        inside = [r for r in rows if window and r[0] is not None and window[0] - 0.1 <= r[0] <= window[1] + 0.1]
        scope = "timed region" if inside else "whole process (no sample fell inside the timed region)"
        for ts, p in (inside or rows):
            try:
                sm.append(float(p[1])); mx.append(float(p[2])); power.append(float(p[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm),
                "scope": scope}


def worker_args(a, result_path="", dump_dir=""):
    from trainingjob_operator_b200.runtime import worker

    d = MODEL_DEFAULTS[a.model]
    argv = ["--model", a.model, "--batch", str(a.batch or d["batch"]), "--seq", str(a.seq or d["seq"] or 1),
            "--steps", str(a.steps), "--warmup", str(a.warmup), "--gemm", a.gemm]
    if a.no_graph:
        argv.append("--no-graph")
    if result_path:
        argv += ["--result", result_path]
    if dump_dir:
        argv += ["--dump-outputs", dump_dir]
    return worker.parse_args(argv), argv


def run_device_timed(a):
    """The ranks the driver launched run the measured loop directly (torchrun env -> our env contract)."""
    from trainingjob_operator_b200.runtime import worker

    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("WORLD_SIZE", "1")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("MASTER_PORT", "29511")
    os.environ.pop("AITJ_MASTER", None)
    rank = int(os.environ["RANK"])
    wa, _ = worker_args(a, dump_dir=a.dump_outputs)
    sampler = ClockSampler() if rank == 0 else None
    if sampler:
        sampler.start()
    res = worker.run(wa)
    clocks = sampler.stop(res.get("timed_region_epoch")) if sampler else None
    return res, clocks


def run_e2e(a, n_gpus):
    """Public-API path: LocalCluster.apply(AITrainingJob) -> controller -> agent -> N worker processes."""
    from trainingjob_operator_b200.cmd.local import LocalCluster

    workdir = tempfile.mkdtemp(prefix="aitj-bench-")
    result_path = os.path.join(workdir, "result.json")
    _, argv = worker_args(a, result_path)
    job = {
        "apiVersion": "elasticdeeplearning.ai/v1", "kind": "AITrainingJob",
        "metadata": {"name": f"bench-{a.model}", "namespace": "default"},
        "spec": {
            "frameworkType": "pytorch", "cleanPodPolicy": "All", "completePolicy": "All", "failPolicy": "Any",
            "replicaSpecs": {"trainer": {
                "replicas": n_gpus, "restartPolicy": "Never",
                "template": {"spec": {"containers": [{
                    "name": "aitj-trainer", "image": "local/aitj-worker",
                    "command": [sys.executable, "-m", "trainingjob_operator_b200.runtime.worker"], "args": argv,
                    "workingDir": ROOT,
                    "env": [{"name": "PYTHONPATH", "value": ROOT}],
                    "resources": {"limits": {"nvidia.com/gpu": 1}}}]}}}}},
    }
    out = {}
    # the node agent's warm pool (agent --warm-pool N): one parked interpreter per GPU slot with torch imported, a live
    # CUDA context and the kernel library loaded -- the steady state of a running daemon, reached before the job arrives
    pool = 0 if a.no_warm_pool else n_gpus
    # gpu_visibility "all": a replica is bound to its GPU by LOCAL_RANK with its peers visible, because the workers'
    # owner-sharded gradient path maps the peers' memory (CUDA symmetric memory needs distinct device indices per rank)
    with LocalCluster(num_gpus=n_gpus, workdir=workdir, warm_pool=pool,
                      gpu_visibility="all" if n_gpus > 1 else "pinned") as lc:
        if pool:
            t_pool = time.time()
            while lc.agent.warm_ready() < pool and time.time() - t_pool < 180:
                time.sleep(0.1)
            out["warm_pool"] = {"size": pool, "ready": lc.agent.warm_ready(), "warm_up_s": round(time.time() - t_pool, 2)}
        t0 = time.time()
        lc.apply(job)
        try:
            running = lc.wait_for_phase(job["metadata"]["name"], ("Running", "Succeed", "Failed"), timeout=300)
            out["reconcile_to_running_s"] = round(time.time() - t0, 3)
            final = lc.wait_for_phase(job["metadata"]["name"], ("Succeed", "Failed", "Timeout", "NodeFail"),
                                      timeout=a.e2e_timeout)
            out["phase"] = final.status.phase
            tr = json.loads(final.annotations.get("aitj.b200/trace", "{}"))
            wt = json.loads(final.annotations.get("aitj.b200/worker-trace", "{}"))
            if tr.get("submitted") and tr.get("running"):
                out["submit_to_all_running_s"] = round(tr["running"] - tr["submitted"], 4)
            if tr.get("submitted") and wt.get("first_step_done"):
                out["submit_to_first_step_s"] = round(wt["first_step_done"] - tr["submitted"], 3)
        except Exception as e:  # noqa: BLE001
            out["error"] = f"{type(e).__name__}: {e}"
            logs = os.path.join(workdir, "logs")
            if os.path.isdir(logs):
                for fn in sorted(os.listdir(logs))[:2]:
                    out.setdefault("log_tail", []).append(open(os.path.join(logs, fn)).read()[-1500:])
    if os.path.exists(result_path):
        out["result"] = json.load(open(result_path))
    return out


def run_torch_stock(a, rank):
    """Comparator arm (baseline/torch_stock.py): stock nn.Module + DDP + fused AdamW + SDPA under bf16 autocast, eager
    or torch.compile-d -- what a user container launched by the reference operator would run.  No repo code on its path."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("aitj_torch_stock", os.path.join(ROOT, "baseline", "torch_stock.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    d = MODEL_DEFAULTS["gpt2"]
    sampler = ClockSampler() if rank == 0 else None
    if sampler:
        sampler.start()
    t0 = time.time()
    r = mod.run(a.batch or d["batch"], a.seq or d["seq"], a.steps, a.warmup, compiled=a.impl.endswith("compiled"))
    t1 = time.time()
    clocks = sampler.stop((t1 - r["ms_per_step"] * a.steps / 1e3 - 0.05, t1)) if sampler else None
    if rank != 0:
        return 0
    line = {
        "metric": "samples/sec (whole job, device-timed CUDA events, max over ranks) of the launched DDP training job",
        "value": r["samples_per_sec"], "unit": "samples/sec", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 autocast (fp32 master weights)", "data": "synthetic tokens / random-init weights (no network)",
        "impl": a.impl,
        "config": {"model": d["name"], "global_batch": r["global_batch"], "per_gpu_batch": r["batch_per_gpu"],
                   "seq_len": r["seq_len"], "parallelism": f"dp{a.gpus}", "params": r["params"],
                   "stack": "nn.Module + DistributedDataParallel + torch.optim.AdamW(fused=True) + SDPA"
                            + (" + torch.compile" if r["compiled"] else " (eager)") + ", grad-clip 1.0",
                   "torch": r["torch"], "warmup_wall_s": r["warmup_wall_s"],
                   "loss_first": r["loss_first"], "loss_last": r["loss_last"],
                   "repo_native_code_mapped": r["repo_native_code_mapped"]},
        "clocks": clocks,
        "e2e": {"value": r["samples_per_sec"], "unit": "samples/sec", "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                "d2h_bytes_per_step": r["d2h_bytes_per_step"],
                "note": "the timed loop itself copies tokens from pinned memory and reads the loss back every step"},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_stock", "torch_stock_compiled"])
    ap.add_argument("--model", default="gpt2", choices=sorted(MODEL_DEFAULTS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default per model)")
    ap.add_argument("--seq", type=int, default=0)
    ap.add_argument("--gemm", default="tcgen05", choices=["tcgen05", "cublas"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-warm-pool", action="store_true", help="e2e arm: cold worker start instead of the agent's warm pool")
    ap.add_argument("--e2e-timeout", type=float, default=900.0)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the last timed step's loss and a sample of the trained state to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(3, a.warmup)

    if a.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable":
                          "reference is a Go Kubernetes operator (no setup.py/pyproject, no GPU code): pip install "
                          "fails and there is no Go toolchain / kube-apiserver in this image (see DESIGN.md)"}))
        return 0

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if a.impl.startswith("torch_stock") and (a.gpus == world or a.gpus == 1):
        return run_torch_stock(a, rank)
    if a.gpus != world and world == 1 and a.gpus > 1:
        # launched without torchrun: spawn the ranks ourselves so `python bench.py --gpus N` also works
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)

    d = MODEL_DEFAULTS[a.model]
    res, clocks = run_device_timed(a)
    # per user: the flag outlives the run, and another user's flag in a shared temp directory can be neither removed nor
    # overwritten
    done_flag = os.path.join(tempfile.gettempdir(),
                             f"aitj_bench_done_{os.getuid()}_{os.environ.get('MASTER_PORT', '0')}")
    if rank != 0:
        # keep the process (and torchrun) alive while rank 0 measures the end-to-end path
        import torch

        torch.cuda.empty_cache()
        t_end = time.time() + a.e2e_timeout + 600
        while not os.path.exists(done_flag) and time.time() < t_end:
            time.sleep(0.5)
        return 0

    import torch

    torch.cuda.empty_cache()
    e2e = {"value": None}
    if not a.no_e2e:
        try:
            if os.path.exists(done_flag):
                os.remove(done_flag)
            o = run_e2e(a, a.gpus)
            r = o.get("result") or {}
            e2e = {"value": r.get("samples_per_sec"), "unit": "samples/sec",
                   "h2d_bytes_per_step": (r.get("h2d_bytes_per_step") or 0) * a.gpus,
                   "d2h_bytes_per_step": (r.get("d2h_bytes_per_step") or 0) * a.gpus,
                   "ms_per_step": r.get("ms_per_step"), "allreduce": r.get("allreduce"),
                   "cuda_graph": r.get("cuda_graph"), "path": "LocalCluster.apply(AITrainingJob) -> operator -> "
                   "agent -> worker processes", **{k: v for k, v in o.items() if k != "result"}}
        finally:
            open(done_flag, "w").write("done")
    else:
        open(done_flag, "w").write("done")

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    flops = res.get("flops_per_step", 0.0) * a.gpus
    ms = res["ms_per_step"]
    line = {
        "metric": "samples/sec (whole job, device-timed CUDA events, max over ranks) of the launched DDP training job",
        "value": res["samples_per_sec"], "unit": "samples/sec", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic tokens / random-init weights (no network)", "impl": "ours",
        "config": {"model": d["name"], "global_batch": res["global_batch"], "per_gpu_batch": res["batch_per_gpu"],
                   "seq_len": res["describe"].get("seq_len"), "parallelism": f"dp{a.gpus}",
                   "params": res["describe"].get("params"), "gemm": res["describe"].get("gemm"),
                   "optimizer": "AdamW (fused flat sweep, fp32 master + bf16 compute copy), grad-clip 1.0",
                   "cuda_graph": res.get("cuda_graph"), "graph_error": res.get("graph_error"),
                   "allreduce": res.get("allreduce"),
                   "l2": "working set (params+activations >> 126 MB L2) exceeds L2; inputs change every step",
                   "loss_first": res.get("loss_first"), "loss_last": res.get("loss_last")},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": res.get("gpu_launches"),
        "launches_per_step": res.get("launches_per_step"),
        "tokens_per_sec": res["samples_per_sec"] * (res["describe"].get("seq_len") or 1),
        "model_tflops": flops / (ms / 1e3) / 1e12 if flops else None,
        "mfu_of_measured_bf16_sustained": (flops / (ms / 1e3) / 1e12 / (peaks.get("bf16_tflops_sustained", 1451.7) * a.gpus))
        if flops else None,
    }
    print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
