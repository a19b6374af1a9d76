"""Worker-side pieces that run on CPU: flat parameter storage, bucketed all-reduce over gloo (2 processes),
LR schedule, env parsing, the flat DDP wrapper (SURVEY.md §4: multi-process paths use gloo, world_size>1)."""
import os
import subprocess
import sys
import textwrap

import pytest

import torch

from trainingjob_operator_b200.models.flat_params import FlatParams, ParamSpec
from trainingjob_operator_b200.models.gpt2 import GPT2Config, flops_per_token, gpt2_param_specs
from trainingjob_operator_b200.runtime.elastic import rendezvous_from_env
from trainingjob_operator_b200.runtime.trainer import SyntheticTokens, cosine_lr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_flat_params_layout_and_masks():
    fp = FlatParams([ParamSpec("w", (10, 30), True), ParamSpec("b", (30,), False, "zeros"),
                     ParamSpec("g", (5,), False, "ones")], "cpu")
    assert fp.total % 256 == 0 and fp.by_name["b"].offset == 512 and fp.by_name["g"].offset == 768
    assert fp.w32("g").tolist() == [1.0] * 5 and float(fp.w32("b").abs().sum()) == 0
    assert fp.wd_mask.tolist() == [1, 1, 0, 0]
    assert fp.num_parameters() == 335
    assert torch.equal(fp.w16("w").float(), fp.w32("w").bfloat16().float())
    a, b = fp.range_of("w", "b")
    assert (a, b) == (0, 768)
    fp.grad("w").fill_(2.0)
    assert float(fp.g32[:300].sum()) == 600.0
    st = fp.state_dict()
    fp2 = FlatParams([ParamSpec("w", (10, 30), True), ParamSpec("b", (30,), False, "zeros"),
                      ParamSpec("g", (5,), False, "ones")], "cpu", seed=9)
    fp2.load_state_dict(st)
    assert torch.equal(fp2.p32, fp.p32)


def test_gpt2_small_parameter_count_and_flops():
    cfg = GPT2Config.small()
    n = 0
    for s in gpt2_param_specs(cfg):
        k = 1
        for d in s.shape:
            k *= d
        n += k
    assert cfg.padded_vocab == 50304
    assert n == 124_475_904                       # 124M (padded vocab), tied lm_head
    assert 7.5e8 < flops_per_token(cfg, 1024) < 9.5e8


def test_lr_schedule_and_synthetic_tokens(monkeypatch):
    assert cosine_lr(0, 1.0, warmup=10) == 0.1 and cosine_lr(9, 1.0, warmup=10) == 1.0
    assert abs(cosine_lr(10_000, 1.0, warmup=10, total=10_000) - 0.1) < 1e-9
    d = SyntheticTokens(100, 2, 8, n_batches=2, pin=False)
    tok, tgt = d.next()
    assert tok.shape == (16,) and torch.equal(tgt, torch.roll(tok, -1)) and d.bytes_per_step == 2 * 16 * 8
    monkeypatch.setenv("WORLD_SIZE", "4"); monkeypatch.setenv("MASTER_PORT", "1234")
    monkeypatch.setenv("AITJ_RENDEZVOUS_GENERATION", "3")
    assert rendezvous_from_env() == {"world": 4, "port": 1234, "generation": 3}


def test_bucket_allreduce_and_flat_ddp_over_gloo():
    script = textwrap.dedent("""
        import os, sys, torch, torch.distributed as dist
        sys.path.insert(0, %r)
        from trainingjob_operator_b200.parallel.ddp import BucketAllReducer, broadcast_state
        from trainingjob_operator_b200.parallel.flat_ddp import FlatDDP
        from trainingjob_operator_b200.models.mnist_cnn import MLP
        rank = int(os.environ["RANK"]); dist.init_process_group("gloo")
        flat = torch.full((1024,), float(rank + 1))
        r = BucketAllReducer(flat, [("a", 512, 1024), ("b", 256, 512), ("c", 0, 256)], backend="gloo", min_bucket_bytes=0)
        for name in ("a", "b", "c"):
            r.hook(name)
        r.wait()
        assert torch.all(flat == 3.0), flat[:4]
        torch.manual_seed(0)
        m = MLP()
        ddp = FlatDDP(m, bucket_bytes=1 << 12, backend="gloo", lr=0.1, optimizer="sgd")
        broadcast_state(ddp.state_tensors(), 0)
        torch.manual_seed(10 + rank)
        x, y = torch.randn(8, 64), torch.randint(0, 10, (8,))
        before = ddp.p32.clone()
        loss = torch.nn.functional.cross_entropy(m(x), y); loss.backward()
        ddp.finish_backward()
        g = ddp.g32.clone()
        ddp.step()
        gl = [torch.zeros_like(g) for _ in range(2)]
        dist.all_gather(gl, g)
        assert torch.allclose(gl[0], gl[1])                 # both ranks hold the same (summed) gradient
        pl = [torch.zeros_like(ddp.p32) for _ in range(2)]
        dist.all_gather(pl, ddp.p32)
        assert torch.allclose(pl[0], pl[1]) and not torch.allclose(pl[0], before)
        assert float(ddp.g32.abs().sum()) == 0.0            # grads zeroed by the optimizer sweep
        print("OK", rank)
        dist.destroy_process_group()        # else gloo's threads can still be joinable at exit ("terminate called ...")
    """ % ROOT)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29733")
        procs.append(subprocess.Popen([sys.executable, "-c", script], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("OK" in o for o in outs)


def test_state_source_is_elected_not_assumed_to_be_rank0():
    """After a re-rendezvous the rank with the most optimizer steps hands its state to everybody (ties: lowest rank);
    a joiner that only has warm-up state never wins -- rank 0 itself may be the replica that was replaced."""
    script = textwrap.dedent("""
        import os, sys, torch, torch.distributed as dist
        sys.path.insert(0, %r)
        from trainingjob_operator_b200.runtime.worker import sync_state
        rank = int(os.environ["RANK"]); dist.init_process_group("gloo")

        class A:
            def __init__(self, steps, fill):
                self.step_count = steps
                self.t = torch.full((16,), float(fill))
            def state_tensors(self): return [self.t]
            def after_state_load(self): pass

        dev = torch.device("cpu")
        # rank 0 is a fresh replacement (warm-up steps only, have_state False); ranks 1 and 2 survived at step 40
        a = A(2 if rank == 0 else 40, rank)
        loop = sync_state(a, 0 if rank == 0 else 45, dev, have_state=rank != 0)
        assert loop == 45 and a.step_count == 40 and float(a.t[0]) == 1.0, (rank, loop, a.step_count, a.t[0])
        # a restarted rank that loaded an older checkpoint loses against the survivors
        a = A(30 if rank == 1 else 50, rank)
        loop = sync_state(a, 30 if rank == 1 else 50, dev)
        assert loop == 50 and a.step_count == 50 and float(a.t[0]) == 0.0
        # nobody has state (fresh start / restart without checkpoint): rank 0 seeds everybody
        a = A(2, rank + 5)
        loop = sync_state(a, 0, dev, have_state=False)
        assert float(a.t[0]) == 5.0
        print("OK", rank)
        dist.destroy_process_group()
    """ % ROOT)
    procs = []
    for rank in range(3):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE="3", MASTER_ADDR="127.0.0.1", MASTER_PORT="29735")
        procs.append(subprocess.Popen([sys.executable, "-c", script], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs


def test_flat_ddp_discards_a_step_that_lost_its_allreduce():
    from trainingjob_operator_b200.models.mnist_cnn import MLP
    from trainingjob_operator_b200.parallel.flat_ddp import FlatDDP

    torch.manual_seed(0)
    m = MLP()
    ddp = FlatDDP(m, backend="gloo", lr=0.1, optimizer="sgd")
    x, y = torch.randn(8, 64), torch.randint(0, 10, (8,))
    torch.nn.functional.cross_entropy(m(x), y).backward()
    assert float(ddp.g32.abs().sum()) > 0
    before = ddp.p32.clone()
    ddp.discard_step()
    assert float(ddp.g32.abs().sum()) == 0.0 and torch.equal(ddp.p32, before)
    assert all(p.grad is not None and p.grad.data_ptr() >= ddp.g32.data_ptr() for p in m.parameters())
    torch.nn.functional.cross_entropy(m(x), y).backward()       # the next step accumulates from zero again
    ddp.finish_backward()
    ddp.step()
    assert not torch.equal(ddp.p32, before)


def test_staged_join_gates_scale_up_until_joiners_announce(monkeypatch):
    """Survivors adopt a larger world only after every joiner announced readiness for that generation (or the
    timeout passed); scale-down and same-size generations are adopted at once."""
    import json
    import time

    from trainingjob_operator_b200.runtime import elastic as E

    state = {"gen": 1, "world": 2, "ann": {}}

    class FakeTransport:
        def __init__(self, *a, **k):
            self.patches = []

        def get(self, info, ns, name):
            return {"metadata": {"annotations": dict(state["ann"])},
                    "status": {"rendezvous": {"generation": state["gen"], "worldSizes": {"trainer": state["world"]},
                                              "masterPort": 1234}}}

        def patch(self, info, ns, name, body):
            self.patches.append(body)
            state["ann"].update(body["metadata"]["annotations"])

    import trainingjob_operator_b200.store.transport as T

    monkeypatch.setattr(T, "HTTPTransport", FakeTransport)
    w = E.ElasticWatcher("http://x", "default", "job", "trainer", generation=1, poll=0.01, world=2)
    try:
        dev = torch.device("cpu")
        time.sleep(0.05)
        assert w.agree(dev) is None                       # nothing new
        state.update(gen=2, world=4)                      # scale up 2 -> 4: ranks 2 and 3 are joiners
        time.sleep(0.1)
        assert w.agree(dev) is None                       # gated: nobody announced yet
        state["ann"][E.ANN_READY_PREFIX + "2"] = json.dumps(2)
        time.sleep(0.1)
        assert w.agree(dev) is None                       # rank 3 still missing
        state["ann"][E.ANN_READY_PREFIX + "3"] = json.dumps(1)   # stale announcement of an older generation
        time.sleep(0.1)
        assert w.agree(dev) is None
        w.announce_ready(3, 2)                            # what the joiner calls; goes through the same annotation
        time.sleep(0.1)
        t = w.agree(dev)
        assert t is not None and t["generation"] == 2 and t["world"] == 4 and t["port"] == 1234
        assert t["observed_at"] <= time.time() - 0.3      # latency is counted from when the change was first seen
        w.adopted(2, 4)
        state.update(gen=3, world=2)                      # scale down: no joiners, adopted at once
        time.sleep(0.1)
        t = w.agree(dev)
        assert t is not None and t["generation"] == 3 and t["world"] == 2
        w.adopted(3, 2)
        w.ready_timeout = 0.15
        state.update(gen=4, world=3)                      # a joiner that never shows up cannot block forever
        time.sleep(0.05)
        assert w.agree(dev) is None
        time.sleep(0.3)
        assert w.agree(dev)["generation"] == 4
    finally:
        w.stop()


def test_generation_agreement_is_a_guarded_collective(monkeypatch):
    """The per-step MAX all-reduce of the newest generation is where a survivor sits when its peer died right after
    a step: it must count as "inside a step" for the StallBreaker, and an abort while it is in flight must surface
    as the same RuntimeError as an aborted training step (4-rank NCCL recovery hung here)."""
    from trainingjob_operator_b200.runtime import elastic as E

    class FakeTransport:
        def __init__(self, *a, **k):
            pass

        def get(self, info, ns, name):
            return {"metadata": {}, "status": {"rendezvous": {"generation": 1, "worldSizes": {"trainer": 2},
                                                              "masterPort": 1}}}

    import trainingjob_operator_b200.store.transport as T

    monkeypatch.setattr(T, "HTTPTransport", FakeTransport)

    class Guard:
        in_step = False
        tripped = False

    g = Guard()
    seen = []

    def fake_all_reduce(t, op=None):
        seen.append(g.in_step)
        if len(seen) == 2:
            g.tripped = True            # the breaker aborted the communicator while we were blocked

    monkeypatch.setattr(E.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(E.dist, "get_world_size", lambda: 2)
    monkeypatch.setattr(E.dist, "all_reduce", fake_all_reduce)
    w = E.ElasticWatcher("http://x", "default", "job", "trainer", generation=1, poll=0.01, world=2)
    try:
        assert w.agree(torch.device("cpu"), guard=g) is None
        assert seen == [True] and g.in_step is False
        with pytest.raises(RuntimeError, match="aborted"):
            w.agree(torch.device("cpu"), guard=g)
        assert g.in_step is False
    finally:
        w.stop()


def test_stall_breaker_only_trips_inside_a_step_with_a_newer_generation_pending(monkeypatch):
    """runtime/rendezvous.py StallBreaker, action="abort": (a) a newer generation is published, (b) the rank has been
    inside one step for longer than the threshold -- both are needed; a rank waiting at a rendezvous is left alone."""
    import time

    from trainingjob_operator_b200.runtime import rendezvous as R

    class Watcher:
        gen = 1

        def fetch_now(self):
            return {"generation": self.gen, "world": 2, "port": 1}

    torn = []
    monkeypatch.setattr(R.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(R, "teardown_group", lambda broken=False: torn.append(broken))
    w = Watcher()
    b = R.StallBreaker(w, after_s=0.2)
    try:
        b.progress(1)
        b.in_step = True
        time.sleep(1.0)
        assert not b.tripped and not torn               # stuck for long, but nothing newer is pending
        w.gen = 2
        b.in_step = False
        b.last_progress = time.time() - 10
        time.sleep(1.0)
        assert not b.tripped and not torn               # newer generation, but not inside a step (e.g. at a rendezvous)
        b.in_step = True
        deadline = time.time() + 3
        while not b.tripped and time.time() < deadline:
            time.sleep(0.05)
        assert b.tripped and torn == [True]
        time.sleep(0.7)
        assert torn == [True]                           # once per trip
    finally:
        b.stop()


def test_stall_exit_leaves_with_137_and_records_it(tmp_path):
    """action="exit" (jobs that cannot recover in place): the stuck rank leaves like the agent's hang detection would --
    exit code 137, written to $AITJ_EXIT_FILE for an adopting agent -- as soon as the controller is repairing the job."""
    exit_file = tmp_path / "exit"
    code = textwrap.dedent("""
        import time
        import torch.distributed as dist
        from trainingjob_operator_b200.runtime import rendezvous as R
        dist.is_initialized = lambda: True
        class W:
            def fetch_now(self):
                return {"generation": 2, "world": 2, "port": 1}
        b = R.StallBreaker(W(), after_s=0.1, action="exit")
        b.progress(1)
        b.in_step = True
        time.sleep(5)
        print("still here")
    """)
    env = dict(os.environ, AITJ_EXIT_FILE=str(exit_file), PYTHONPATH=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 137, (r.returncode, r.stdout, r.stderr)
    assert "still here" not in r.stdout and "does not recover in place" in r.stdout
    assert exit_file.read_text() == "137"


def test_zygote_command_parsing():
    from trainingjob_operator_b200.runtime.zygote import split_python_command as sp

    assert sp(["python", "-m", "pkg.mod", "--a", "1"]) == ("module", "pkg.mod", ["--a", "1"])
    assert sp(["/usr/bin/python3", "-u", "train.py", "x"]) == ("script", "train.py", ["x"])
    assert sp(["python", "-c", "print(1)"]) is None
    assert sp(["/bin/sh", "-c", "true"]) is None
    assert sp(["python"]) is None and sp([]) is None


def test_async_checkpoint_is_a_consistent_snapshot_and_never_blocks_on_a_busy_writer(tmp_path, monkeypatch):
    from trainingjob_operator_b200.runtime import checkpoint as ck

    path = str(tmp_path / "job.pt")
    w = ck.AsyncCheckpointer(path)
    a, b = torch.arange(1000, dtype=torch.float32), torch.ones(7, 3)
    assert ck.load_into(path, [a, b]) is None                    # nothing there yet
    assert w.save(10, [a, b], extra={"world": 2})
    a.add_(1.0)                                                  # the step loop moves on while the file is written
    assert w.wait(30)
    x, y = torch.zeros(1000), torch.zeros(7, 3)
    meta = ck.load_into(path, [x, y])
    assert meta == {"step": 10, "world": 2}
    assert torch.equal(x, torch.arange(1000, dtype=torch.float32)) and torch.equal(y, b)   # state as of save()
    assert not os.path.exists(path + ".tmp")

    # a slow disk: the next interval's checkpoint is skipped, not queued, and the old file stays readable
    gate = __import__("threading").Event()
    real_save = torch.save

    def slow_save(obj, f):
        gate.wait(30)
        real_save(obj, f)

    monkeypatch.setattr(torch, "save", slow_save)
    assert w.save(20, [a, b])
    assert w.busy() and w.save(30, [a, b]) is False and w.stats["skipped_busy"] == 1
    assert ck.load_into(path, [x, y])["step"] == 10              # readers never see a torn / half-written file
    gate.set()
    assert w.wait(30) and ck.load_into(path, [x, y])["step"] == 20 and w.stats["saved"] == 2

    # a checkpoint of another architecture is refused, not half-loaded
    try:
        ck.load_into(path, [torch.zeros(5)])
        raise AssertionError("mismatch accepted")
    except ValueError as e:
        assert "does not match" in str(e)

    # a failed write surfaces on the next call instead of vanishing in the thread
    monkeypatch.setattr(torch, "save", lambda obj, f: (_ for _ in ()).throw(OSError("disk full")))
    assert w.save(40, [a, b])
    try:
        w.wait(30)
        raise AssertionError("write error swallowed")
    except RuntimeError as e:
        assert "disk full" in str(e)


def test_gathering_ranks_is_bounded_and_ends_early_on_a_newer_generation(tmp_path):
    """Two of three ranks wait on a generation's store.  (a) The moment a newer generation is published they stop
    waiting (StaleGeneration) instead of sitting out the attempt; (b) without one they give up at the attempt deadline;
    (c) with all ranks present the group forms and works."""
    script = textwrap.dedent("""
        import os, sys, time, torch, torch.distributed as dist
        sys.path.insert(0, %r)
        from trainingjob_operator_b200.runtime import worker as W
        rank, world, port = int(os.environ["RANK"]), int(os.environ["WORLD"]), int(os.environ["PORT"])
        flag = os.environ["FLAG"]
        dev = torch.device("cpu")
        t0 = time.time()
        try:
            W.init_process_group(rank, world, port, dev, timeout_s=20, attempt_timeout_s=float(os.environ["ATTEMPT"]),
                                 stale=lambda: os.path.exists(flag))
        except W.StaleGeneration:
            print("STALE %%.2f" %% (time.time() - t0)); sys.exit(0)
        except TimeoutError:
            print("TIMEOUT %%.2f" %% (time.time() - t0)); sys.exit(0)
        except Exception as e:            # the store's host saw the newer generation first and closed the store
            print("LOST %%.2f %%s" %% (time.time() - t0, type(e).__name__)); sys.exit(0)
        t = torch.ones(1) * (rank + 1)
        dist.all_reduce(t)
        print("SUM %%d" %% int(t[0]))
        dist.destroy_process_group()
    """ % ROOT)

    def launch(ranks, world, port, attempt, flag):
        procs = []
        for r in ranks:
            env = dict(os.environ, RANK=str(r), WORLD=str(world), PORT=str(port), ATTEMPT=str(attempt), FLAG=flag)
            procs.append(subprocess.Popen([sys.executable, "-c", script], env=env, stdout=subprocess.PIPE,
                                          stderr=subprocess.STDOUT, text=True))
        return procs

    import time
    flag = str(tmp_path / "newer-generation")
    # (a) rank 2 never comes; the newer generation appears after ~2 s of a 60 s attempt
    procs = launch([0, 1], 3, 29741, 60, flag)
    time.sleep(6.0)                       # interpreter start + torch import, then they wait on the store
    open(flag, "w").close()
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert "STALE" in outs[0] and ("STALE" in outs[1] or "LOST" in outs[1]), outs
    assert float(outs[0].split("STALE")[1].split()[0]) < 30, outs      # its own clock: not the 60 s attempt
    os.unlink(flag)
    # (b) bounded by the attempt when nothing else happens
    outs = [p.communicate(timeout=90)[0] for p in launch([0, 1], 3, 29742, 3, flag)]
    assert "TIMEOUT" in outs[0] and ("TIMEOUT" in outs[1] or "LOST" in outs[1]), outs     # (host gone first: LOST)
    assert float(outs[0].split("TIMEOUT")[1].split()[0]) < 10, outs
    # (c) everybody present
    outs = [p.communicate(timeout=90)[0] for p in launch([0, 1, 2], 3, 29743, 30, flag)]
    assert all("SUM 6" in o for o in outs), outs


def test_owner_shard_bounds_are_balanced_and_aligned():
    """Ownership bounds of the flat gradient space (parallel/symm.py): ascending, every bound a multiple of 256 elements
    (the AdamW sweep's weight-decay blocks) and of 32 rows of the 2-D tensor it falls into (the wgrad epilogue sends
    32-row groups to one owner), shares within a few percent of 1/N."""
    from trainingjob_operator_b200.models.bert import BertConfig, bert_param_specs
    from trainingjob_operator_b200.models.flat_params import FlatParams
    from trainingjob_operator_b200.models.gpt2 import GPT2Config, gpt2_param_specs
    from trainingjob_operator_b200.parallel.symm import shard_bounds

    for specs in (gpt2_param_specs(GPT2Config.small()), gpt2_param_specs(GPT2Config.tiny()),
                  bert_param_specs(BertConfig.base())):
        P = FlatParams(specs, "cpu", with_optimizer_state=False)
        for world in (2, 3, 4, 8):
            b = shard_bounds(P.specs, P.total, world)
            assert len(b) == world + 1 and b[0] == 0 and b[-1] == P.total and b == sorted(b)
            for x in b[1:-1]:
                assert x % 256 == 0
                s = next(s for s in P.specs if s.offset <= x <= s.offset + s.padded)
                if len(s.shape) == 2 and s.offset < x < s.offset + s.numel:
                    assert (x - s.offset) % (32 * s.shape[1]) == 0, (s.name, x)
            shares = [(b[i + 1] - b[i]) * world / P.total for i in range(world)]
            assert 0.9 < min(shares) and max(shares) < 1.1, shares


@pytest.mark.parametrize("name,batch,params", [("mnist", 32, 1_199_882), ("resnet50", 2, 25_557_032)])
def test_nn_module_workers_step_on_cpu(name, batch, params):
    """BASELINE configs 2 and 3 (MNIST CNN, ResNet-50 -- own definition, the canonical 25,557,032 parameters) through the
    worker's nn.Module adapter: flat parameter / gradient buffers, fused optimizer sweep, state hand-off tensors."""
    import types

    from trainingjob_operator_b200.runtime import worker as W

    args = types.SimpleNamespace(seed=0, lr=1e-3, no_graph=True, gemm="tcgen05")
    ad = W.TorchAdapter(name, batch, args, torch.device("cpu"))
    ad.bind(None)
    assert sum(p.numel() for p in ad.module.parameters()) == params
    losses = [float(ad.train_step()) for _ in range(2)]
    assert all(l == l and abs(l) < 1e4 for l in losses)
    state = ad.state_tensors()
    assert state and all(t.dtype == torch.float32 for t in state)
    snap = [t.clone() for t in state]
    ad.train_step()
    assert any(not torch.equal(a, b) for a, b in zip(snap, state))       # the state tensors ARE the live state
    ad.after_state_load()


def test_bench_dump_outputs_are_the_same_for_the_same_arguments(tmp_path):
    """``bench.py --dump-outputs``: the last timed step's loss and the trained state land as float32 ``.npy`` files within
    64 MB, and two runs with the same arguments write the same values (seeded inputs and initial weights)."""
    import json

    import numpy as np

    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--model", "mnist", "--batch", "8", "--steps",
                            "2", "--warmup", "3", "--no-e2e", "--dump-outputs", str(out)], cwd=str(tmp_path),
                           env=dict(os.environ, OMP_NUM_THREADS="2", CUDA_VISIBLE_DEVICES=""),   # CPU: bitwise repeatable
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2
        dumps.append({f.name: np.load(f) for f in sorted(out.iterdir())})
    a, b = dumps
    assert sorted(a) == ["exp_avg.npy", "exp_avg_sq.npy", "loss.npy", "params.npy"]
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(np.array_equal(a[k], b[k]) for k in a)
