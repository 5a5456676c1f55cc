"""T2: full DecoupledTrainer.train() on 2 CPU ranks over gloo (BASELINE config 1 plumbing)."""
import os
import sys
import tempfile

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, method, tmp, extra, q):
    # every worker hides the GPUs before touching CUDA: these are CPU ranks, and the trainer takes CUDA whenever it sees a device
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(CUDA_VISIBLE_DEVICES="", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    os.chdir(tmp)
    torch.set_num_threads(2)
    from acco_b200 import DecoupledTrainer
    from acco_b200.data import synthetic_pretrain_dataset
    from acco_b200.launch import shutdown_distributed
    from helpers import LOG, base_args, tiny_model
    model = tiny_model(seed=rank)                      # different init per rank: init sync must fix that
    ds = synthetic_pretrain_dataset(300, 30, 96, 16, seed=7)
    args = base_args(method_name=method, nb_steps_tot=48, learning_rate=5e-3, batch_size=4, save=(method == "acco"), **extra)
    t = DecoupledTrainer(model=model, train_dataset=ds, args=args, log=LOG)
    hetero = extra.get("_hetero")
    if hetero:
        t._hook_extra_microbatches = lambda r, rnd: (1 if r == 0 else 0)   # rank 0 is "faster": more micro-batches per round
    losses = []
    checks = []
    while not t.finished():
        flipped = t.step()
        losses.append(float(t.loss_host))
        if flipped:
            # all ranks must hold identical parameters in the buffer the last finished round wrote
            done_theta = t.arena.theta[(t.sched.round - (1 if t._inflight is not None else 0)) % 2]
            checks.append(float(done_theta.double().sum()))
    t._drain()
    stats = t._finish("")
    q.put((rank, losses[:4], losses[-4:], checks, stats["count_grad_tot"], float(t.params.double().sum()),
           t.sched.opt_steps, t.size_slice, t.size_local_slice, t.len_params))
    shutdown_distributed()


def _run(method, **extra):
    from acco_b200.launch import free_port
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    with tempfile.TemporaryDirectory() as tmp:
        procs = [ctx.Process(target=_worker, args=(r, 2, port, method, tmp, extra, q)) for r in range(2)]
        for p in procs:
            p.start()
        out = [q.get(timeout=240) for _ in procs]
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        files = set(os.listdir(tmp))
        ck = set(os.listdir(os.path.join(tmp, "checkpoints"))) if "checkpoints" in files else set()
    return sorted(out), files, ck


@pytest.mark.parametrize("method", ["acco", "dpu", "ddp"])
def test_two_rank_training(method):
    out, files, ck = _run(method)
    (r0, first0, last0, chk0, tot0, sum0, steps0, sl0, loc0, n0), (r1, first1, last1, chk1, tot1, sum1, steps1, sl1, loc1, n1) = out
    assert tot0 == tot1 >= 48 and steps0 == steps1
    assert chk0 == chk1 and len(chk0) > 3                 # identical parameters on both ranks after every round
    assert sum0 == sum1
    assert sum(last0) / 4 < sum(first0) / 4               # loss goes down
    assert "results.csv" in files                         # rank 0 artefacts only
    if method == "acco":
        assert len(ck) == 1 and next(iter(ck)).endswith("_model.pt") and next(iter(ck)) != "torchrun_model.pt"   # unique run id
    # ragged slice math: N odd or even, last rank may own a short slice
    assert sl0 == sl1 and loc0 + loc1 == n0


def test_heterogeneous_counts_still_consistent():
    out, _, _ = _run("acco", _hetero=True)
    (_, _, _, chk0, tot0, sum0, steps0, *_), (_, _, _, chk1, tot1, sum1, steps1, *_) = out
    assert tot0 == tot1 and steps0 == steps1 and sum0 == sum1 and chk0 == chk1
    # rank 0 contributed 2 micro-batches per phase, rank 1 one: 3 per half-round -> 6 per optimizer step
    assert tot0 % 6 == 0


def test_init_avg_mode_matches_reference_behaviour():
    out, _, _ = _run("acco", init_sync="avg")
    assert out[0][5] == out[1][5]


def _worker3(rank, world, port, tmp, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(CUDA_VISIBLE_DEVICES="", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    os.chdir(tmp)
    torch.set_num_threads(1)
    from acco_b200 import DecoupledTrainer
    from acco_b200.data import synthetic_pretrain_dataset
    from acco_b200.launch import shutdown_distributed
    from helpers import LOG, base_args, tiny_model
    ds = synthetic_pretrain_dataset(300, 30, 96, 16, seed=7)
    out = {}
    for method, extra in (("acco", {}), ("ddp", {"ddp_impl": "torch"}), ("dpu", {"run_expe_slow": True, "slow_ranks": [1], "slow_factor_ms": 2, "lr_unit": "grads"})):
        t = DecoupledTrainer(model=tiny_model(seed=0, hidden=40), train_dataset=ds,
                             args=base_args(method_name=method, nb_steps_tot=36, learning_rate=5e-3, batch_size=2, **extra), log=LOG)
        t.train()
        flat = torch.cat([p.detach().reshape(-1).double() for p in t.model.parameters()])
        out[method] = (t.sched.count_grad_tot, float(flat.sum()), float(t.loss_host), getattr(t, "size_slice", 0), getattr(t, "len_params", 0))
    q.put((rank, out))
    shutdown_distributed()


def test_three_ranks_ragged_slices_all_methods_and_torch_ddp():
    """W=3 does not divide the parameter count (ragged last slice); also exercises ddp_impl='torch'
    (DDP + ZeroRedundancyOptimizer, the reference's baseline), slow-rank injection and lr_unit='grads'."""
    from acco_b200.launch import free_port
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    with tempfile.TemporaryDirectory() as tmp:
        procs = [ctx.Process(target=_worker3, args=(r, 3, port, tmp, q)) for r in range(3)]
        for p in procs:
            p.start()
        res = dict(q.get(timeout=300) for _ in procs)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    for method in ("acco", "ddp", "dpu"):
        tot = {res[r][method][0] for r in range(3)}
        sums = {res[r][method][1] for r in range(3)}
        assert len(tot) == 1 and tot.pop() >= 36, method
        assert len(sums) == 1, (method, sums)              # every rank ends with identical parameters
    sl, n = res[0]["acco"][3], res[0]["acco"][4]
    assert n % 3 != 0 and sl * 3 >= n                      # the configuration really is ragged


def _worker_resume(rank, world, port, tmp, phase, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(CUDA_VISIBLE_DEVICES="", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank), ACCO_RUN_ID="resume")
    os.chdir(tmp)
    torch.set_num_threads(2)
    from acco_b200 import DecoupledTrainer
    from acco_b200.data import synthetic_pretrain_dataset
    from acco_b200.launch import shutdown_distributed
    from helpers import LOG, base_args, tiny_model
    ds = synthetic_pretrain_dataset(300, 30, 96, 16, seed=7)
    ck = os.path.join(tmp, "checkpoints", "resume_model.pt")
    if phase == "first":
        args = base_args(nb_steps_tot=24, learning_rate=5e-3, batch_size=4, save=True, save_optimizer=True, scheduler_name="cosine", warmup=2)
        t = DecoupledTrainer(model=tiny_model(seed=0), train_dataset=ds, args=args, log=LOG)
        t.train()
        q.put((rank, t.sched.count_grad_tot, t.sched.opt_steps, float(t.sharded_optimizer.exp_avg.double().abs().sum())))
    else:
        args = base_args(nb_steps_tot=48, learning_rate=5e-3, batch_size=4, save=False, resume_from=ck, scheduler_name="cosine", warmup=2)
        t = DecoupledTrainer(model=tiny_model(seed=5), train_dataset=ds, args=args, log=LOG)
        restored = (t.sched.count_grad_tot, t.sched.opt_steps, float(t.sharded_optimizer.exp_avg.double().abs().sum()))
        t.train()
        q.put((rank, restored, t.sched.count_grad_tot, float(t.params.double().sum())))
    shutdown_distributed()


def test_two_rank_resume_restores_every_ranks_optimizer_shard():
    """`save_optimizer`: EVERY rank writes its shard (not only rank 0); a 2-rank resume restores Adam state + counters on both
    ranks, finishes on the same round everywhere, and a missing shard is an error instead of a silent cold start."""
    from acco_b200.launch import free_port
    ctx = mp.get_context("spawn")
    with tempfile.TemporaryDirectory() as tmp:
        outs = {}
        for phase in ("first", "second"):
            q = ctx.Queue()
            port = free_port()
            procs = [ctx.Process(target=_worker_resume, args=(r, 2, port, tmp, phase, q)) for r in range(2)]
            for p in procs:
                p.start()
            outs[phase] = sorted(q.get(timeout=240) for _ in procs)
            for p in procs:
                p.join(timeout=60)
                assert p.exitcode == 0
            if phase == "first":
                files = set(os.listdir(os.path.join(tmp, "checkpoints")))
                assert {"resume_model.pt", "resume_model_optim_rank0of2.pt", "resume_model_optim_rank1of2.pt"} <= files, files
        (r0, tot0, steps0, m0), (r1, tot1, steps1, m1) = outs["first"]
        assert tot0 == tot1 >= 24 and steps0 == steps1 and m0 > 0 and m1 > 0
        (_, rest0, fin0, sum0), (_, rest1, fin1, sum1) = outs["second"]
        # both ranks restored the counters and a non-trivial Adam state (their own shard)
        assert rest0[:2] == (tot0, steps0) and rest1[:2] == (tot1, steps1)
        assert abs(rest0[2] - m0) < 1e-9 and abs(rest1[2] - m1) < 1e-9
        assert fin0 == fin1 >= 48 and sum0 == sum1
        # elastic restart: the same checkpoint resumed on THREE ranks and on ONE rank - every rank re-assembles its slice of the new
        # layout from the two old shards; the total Adam state is preserved and the ranks stay in lockstep
        for world in (3, 1):
            q = ctx.Queue()
            port = free_port()
            procs = [ctx.Process(target=_worker_resume, args=(r, world, port, tmp, "second", q)) for r in range(world)]
            for p in procs:
                p.start()
            out = sorted(q.get(timeout=240) for _ in procs)
            for p in procs:
                p.join(timeout=60)
                assert p.exitcode == 0
            assert all(o[1][:2] == (tot0, steps0) for o in out), out
            assert abs(sum(o[1][2] for o in out) - (m0 + m1)) < 1e-6 * (m0 + m1), (out, m0, m1)
            assert len({o[2] for o in out}) == 1 and out[0][2] >= 48 and len({o[3] for o in out}) == 1


def _worker_preempt(rank, world, port, tmp, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(CUDA_VISIBLE_DEVICES="", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank), ACCO_RUN_ID="pre")
    os.chdir(tmp)
    torch.set_num_threads(2)
    from acco_b200 import DecoupledTrainer
    from acco_b200.data import synthetic_pretrain_dataset
    from acco_b200.launch import shutdown_distributed
    from helpers import LOG, base_args, tiny_model
    ds = synthetic_pretrain_dataset(300, 30, 96, 16, seed=7)
    args = base_args(nb_steps_tot=10 ** 6, learning_rate=5e-3, batch_size=4, save=True, save_optimizer=True, save_interval_s=10 ** 6, preempt_save=True)
    t = DecoupledTrainer(model=tiny_model(seed=0), train_dataset=ds, args=args, log=LOG)
    steps = 0
    while not t.finished():
        t.step()
        steps += 1
        if rank == 1 and steps == 9:
            t._stop_requested = True          # what the SIGTERM handler does - on ONE rank only
        assert steps < 400, "the other rank never learned about the pre-emption"
    t._drain()
    t._finish("")
    q.put((rank, t.sched.count_grad_tot, t.sched.count_com, float(t.params.double().sum())))
    shutdown_distributed()


def test_preemption_signal_on_one_rank_stops_every_rank_after_the_same_round():
    from acco_b200.launch import free_port
    ctx = mp.get_context("spawn")
    with tempfile.TemporaryDirectory() as tmp:
        q = ctx.Queue()
        port = free_port()
        procs = [ctx.Process(target=_worker_preempt, args=(r, 2, port, tmp, q)) for r in range(2)]
        for p in procs:
            p.start()
        out = sorted(q.get(timeout=240) for _ in procs)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        (_, tot0, com0, sum0), (_, tot1, com1, sum1) = out
        assert tot0 == tot1 and com0 == com1 and sum0 == sum1 and tot0 < 200
        files = set(os.listdir(os.path.join(tmp, "checkpoints")))
        assert {f"pre_model_{tot0}.pt", f"pre_model_{tot0}_optim_rank0of2.pt", f"pre_model_{tot0}_optim_rank1of2.pt"} <= files, files
        assert "pre_model.pt" not in files            # no "final" checkpoint for a run that was cut short


def _worker_dist_utils(rank, world, port, tmp, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(CUDA_VISIBLE_DEVICES="", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank), ACCO_RUN_ID="du")
    os.chdir(tmp)
    torch.set_num_threads(2)
    from acco_b200 import DecoupledTrainer
    from acco_b200.data import synthetic_pretrain_dataset
    from acco_b200.launch import shutdown_distributed
    from acco_b200.utils.dist import gather_concat, gather_scalars, rank_zero_first, reduce_mean
    from helpers import LOG, base_args, tiny_model
    t = DecoupledTrainer(model=tiny_model(seed=0), train_dataset=synthetic_pretrain_dataset(300, 30, 96, 16, seed=7),
                         eval_dataset=synthetic_pretrain_dataset(80, 30, 96, 16, seed=8), log=LOG,
                         args=base_args(nb_steps_tot=16, batch_size=4, eval=True, eval_step=3, eval_all_ranks=True))
    seen = []
    from acco_b200 import TrainerCallback

    class Rec(TrainerCallback):
        def on_evaluate(self, trainer, eval_loss):
            seen.append(eval_loss)

    t.add_callback(Rec())
    t.train()
    # ragged gather: rank r contributes r + 1 rows
    rows = torch.full((rank + 1, 2), float(rank))
    cat = gather_concat({"a": rows, "b": [torch.tensor(rank)]}, None)
    sc = gather_scalars([rank, rank + 0.5])
    mean = reduce_mean(float("nan") if rank == 0 else 4.0)
    order = []
    with rank_zero_first(rank):
        marker = os.path.join(tmp, "cache.marker")
        order.append(os.path.exists(marker))
        if rank == 0:
            open(marker, "w").write("x")
    q.put((rank, seen, cat["a"].tolist(), cat["b"][0].tolist(), sc.tolist(), mean, order))
    shutdown_distributed()


def test_distributed_helpers_and_all_rank_eval_mean():
    """`utils/dist.py` on 2 gloo ranks: ragged `gather_concat` over nested containers, `gather_scalars`, NaN-skipping `reduce_mean`,
    `rank_zero_first`; `eval_all_ranks=True` reports the same (mean) eval loss on every rank."""
    from acco_b200.launch import free_port
    ctx = mp.get_context("spawn")
    with tempfile.TemporaryDirectory() as tmp:
        q = ctx.Queue()
        port = free_port()
        procs = [ctx.Process(target=_worker_dist_utils, args=(r, 2, port, tmp, q)) for r in range(2)]
        for p in procs:
            p.start()
        out = sorted(q.get(timeout=240) for _ in procs)
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    (_, seen0, a0, b0, sc0, mean0, order0), (_, seen1, a1, b1, sc1, mean1, order1) = out
    assert seen0 and seen0 == seen1                                  # identical mean eval loss on both ranks, at the same rounds
    assert a0 == a1 == [[0.0, 0.0], [1.0, 1.0], [1.0, 1.0]] and b0 == b1 == [0, 1]
    assert sc0 == sc1 == [0.0, 0.5, 1.0, 1.5] and mean0 == mean1 == 4.0
    assert order0 == [False] and order1 == [True]                    # rank 0 ran the body first, rank 1 found its result
