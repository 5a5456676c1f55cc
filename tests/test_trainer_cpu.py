import csv
import os
import types

import numpy as np
import pytest
import torch

from acco_b200 import DecoupledTrainer
from acco_b200.data import synthetic_pretrain_dataset, synthetic_sft_dataset, ByteTokenizer, synthetic_text_dataset
from acco_b200.launch import DistEnv

from helpers import LOG, ToyQuadratic, base_args, tiny_model

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def make(method="acco", model=None, ds=None, **kw):
    ds = ds if ds is not None else synthetic_pretrain_dataset(200, 30, 96, 16, seed=3)
    return DecoupledTrainer(model=model or tiny_model(), train_dataset=ds, args=base_args(method_name=method, **kw), log=LOG,
                            env=DistEnv(id_run="job42"))


@pytest.mark.parametrize("method", ["acco", "dpu", "ddp"])
def test_loss_decreases_and_counters(workdir, method):
    t = make(method, nb_steps_tot=80, learning_rate=5e-3, batch_size=4)
    first = None
    losses = []
    while not t.finished():
        t.step()
        losses.append(float(t.loss_host))
    stats = t._finish("")
    assert stats["count_grad_tot"] >= 80
    assert sum(losses[-10:]) / 10 < sum(losses[:10]) / 10 - 0.2
    if method == "acco":
        assert t.sched.opt_steps == t.sched.count_com // 2
    else:
        assert t.sched.opt_steps == t.sched.count_com


def test_train_api_and_artefacts(workdir):
    t = make("acco", save=True, tensorboard=True, nb_steps_tot=8)
    t.run_name = "r"
    stats = t.train()
    assert stats["backend"] == "gloo"
    # checkpoint layout + HF key names (trainer_decoupled.py:594-598)
    path = workdir / "checkpoints" / "job42_model.pt"
    assert path.exists()
    sd = torch.load(path)
    assert "model.layers.0.self_attn.q_proj.weight" in sd and "lm_head.weight" in sd
    assert sd["model.embed_tokens.weight"].shape == (96, 32)
    # results.csv: args + the reference's extra columns (utils/logs_utils.py:57-66)
    rows = list(csv.DictReader(open(workdir / "results.csv")))
    assert len(rows) == 1
    for k in ("0_id_run", "Tot_time", "N_workers", "n_nodes", "cuda_device", "Loss_final", "method_name", "learning_rate"):
        assert k in rows[0]
    assert rows[0]["0_id_run"] == "job42" and rows[0]["N_workers"] == "1"
    assert (workdir / "tensorboard").exists()


def test_results_csv_column_union(workdir):
    from acco_b200.obs import save_result
    save_result("r.csv", {"a": 1, "b": 2})
    save_result("r.csv", {"b": 3, "c": 4})
    rows = list(csv.DictReader(open("r.csv")))
    assert rows[0] == {"a": "1", "b": "2", "c": ""} and rows[1] == {"a": "", "b": "3", "c": "4"}


def test_dpu_and_ddp_checkpoint_names(workdir):
    make("dpu", save=True, nb_steps_tot=4).train()
    make("ddp", save=True, nb_steps_tot=4).train()
    names = sorted(os.listdir(workdir / "checkpoints"))
    assert names == ["job42_ddp_model.pt", "job42dpu_model.pt"]       # sic: the reference's DPU name has no underscore


def test_acco_equals_large_batch_ddp_when_estimate_is_exact(workdir):
    """T1(c): with lr tiny the tentative theta~ == theta to fp32 precision is not guaranteed, so force
    it: a model whose gradient does not depend on theta (linear loss).  Then one ACCO real step
    (g~ + g over 2 micro-batches) must equal one DDP step with n_grad_accumulation=2 bit-for-bit."""
    class Lin(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.linspace(-1, 1, 10))

        def forward(self, input_ids=None, labels=None, **kw):
            x = input_ids.float().mean(0)[:10] / 50.0
            return ((self.w * x).sum(),)

    ds = synthetic_pretrain_dataset(100, 30, 96, 16, seed=5)
    ta = make("acco", model=Lin(), ds=ds, nb_steps_tot=8, learning_rate=1e-1, weight_decay=0.1)
    td = make("ddp", model=Lin(), ds=ds, nb_steps_tot=8, learning_rate=1e-1, weight_decay=0.1, n_grad_accumulation=2)
    ta.train()
    td.train()
    assert ta.sched.opt_steps == td.sched.opt_steps == 4
    assert torch.equal(ta.sharded_optimizer.master, td.sharded_optimizer.master)
    assert torch.equal(ta.model.w.detach(), td.model.w.detach())


def test_golden_trace_against_reference_step_functions(workdir):
    """T1(a): our trainer against the trace of the original ACCO implementation on the same toy, stored in
    `golden/acco_reference_trace.npy` (float32, one row of parameters per flip).  The trace was produced by the original's own
    `communication_step` / `update_buffers_step` (CPU, gloo W=1, AdamW(capturable=False), lr 0.1, betas (0.9, 0.95), no weight
    decay, constant LR) from p0 = [1, 2, 3, 4] with gradient 0.1*(k+1)*p at the k-th evaluation: g0 at p0 fills the first
    communication buffer, then each of 6 rounds runs one micro-batch while it communicates.  Parameters after every flip must agree."""
    p0 = [1.0, 2.0, 3.0, 4.0]
    lr = 0.1
    ref_trace = torch.from_numpy(np.load(os.path.join(GOLDEN, "acco_reference_trace.npy")))
    assert ref_trace.shape == (6, 4) and ref_trace.dtype == torch.float32

    t = make("acco", model=ToyQuadratic(p0), nb_steps_tot=10 ** 6, learning_rate=lr, reference_quirks=True,
             adam_beta1=0.9, adam_beta2=0.95)
    ours = []
    t.step()                                                     # priming phase (g~0) + launch round 0
    for r in range(6):
        t.step()                                                 # phase during round r, then flip
        t._bind_compute_buffers()
        ours.append(t.params.detach().clone())
    for r, (a, b) in enumerate(zip(ref_trace, ours)):
        torch.testing.assert_close(b, a, rtol=1e-6, atol=1e-7, msg=f"round {r}: ours {b} vs reference {a}")
    # the SURVEY table (first component, 4 decimals)
    assert [round(float(x[0]), 4) for x in ours] == [0.9, 0.9014, 0.8072, 0.8095, 0.7172, 0.7183]
    assert t.sched.count_grad_tot == 6 and t.sched.opt_steps == 3 + 1     # +1: the Q1 state-only commit of round 0


def test_clean_mode_differs_from_quirk_only_in_adam_state(workdir):
    t = make("acco", model=ToyQuadratic([1.0, 2.0, 3.0, 4.0]), nb_steps_tot=10 ** 6, learning_rate=0.1,
             adam_beta1=0.9, adam_beta2=0.999)
    t.step()                                   # priming + round 0 (tentative; executes synchronously on CPU)
    assert float(t.arena.theta[1][0]) == pytest.approx(0.9, abs=1e-6)   # theta~1: a first Adam step moves by lr
    assert t.sharded_optimizer.step == 0                                 # ... and leaves no trace in the state
    assert float(t.sharded_optimizer.master[0]) == 1.0 and t.sharded_optimizer.exp_avg.abs().sum() == 0
    t.step()                                   # phase on theta0, flip, round 1 (real)
    assert t.sharded_optimizer.step == 1
    assert float(t.arena.theta[0][0]) == pytest.approx(0.9, abs=1e-6)   # clean real step 1 is again a *first* Adam step
    assert float(t.sharded_optimizer.master[0]) == pytest.approx(0.9, abs=1e-6)


def test_warmup_then_acco(workdir):
    t = make("acco", n_warmup_steps=3, nb_steps_tot=14)
    t.train()
    s = t.sched
    assert s.opt_steps == 3 + (s.count_com - 3) // 2 and s.count_grad_tot >= 14


def test_dynamic_accumulation_counts(workdir):
    """If the round is not finished the next phase accumulates more; the global count normalises."""
    t = make("acco", nb_steps_tot=10 ** 6)
    t._hook_extra_microbatches = lambda rank, rnd: 2 if rnd % 2 == 1 else 0
    t.step(); t.step(); t.step()
    # round 1 (real) consumed stash (1 micro-batch) + acc (1+0): phase during round 0 has rnd==1 -> 3 micro-batches
    assert t.sched.count_grad_tot == 1 + 3


def test_sft_padded_batches_and_eval(workdir):
    ds = synthetic_sft_dataset(120, 10, 96, 16, seed=1)
    ev = synthetic_sft_dataset(40, 10, 96, 16, seed=2)
    tok = ByteTokenizer()
    tok.pad_token_id = tok.eos_token_id = 95
    t = DecoupledTrainer(model=tiny_model(), tokenizer=tok, train_dataset=ds, eval_dataset=ev,
                         args=base_args(const_len_batch=False, nb_steps_tot=12, eval=True, eval_step=3, n_grad_accumulation=2),
                         log=LOG, env=DistEnv(id_run="sft"))
    t.train()
    assert t.sched.count_grad_tot >= 12
    el = t.eval_loop()
    assert torch.isfinite(el)


def test_text_dataset_is_tokenized(workdir):
    tok = ByteTokenizer()
    ds = synthetic_text_dataset(200, 30, seed=0)
    m = tiny_model(vocab=257)
    t = DecoupledTrainer(model=m, tokenizer=tok, train_dataset=ds, args=base_args(nb_steps_tot=4), log=LOG, env=DistEnv())
    assert t.train_dataset.column_names == ["input_ids"]
    t.train()


def test_checkpoint_resume(workdir):
    a = dict(save=True, save_optimizer=True, nb_steps_tot=10)
    t = make("acco", **a)
    t.train()
    ck = str(workdir / "checkpoints" / "job42_model.pt")
    t2 = make("acco", resume_from=ck, **a)
    assert t2.sharded_optimizer.step == t.sharded_optimizer.step > 0
    assert torch.equal(t2.sharded_optimizer.exp_avg, t.sharded_optimizer.exp_avg)
    torch.testing.assert_close(t2.params, t.params)
    assert t2.sched.opt_steps == t.sched.opt_steps and t2.sched.count_grad_tot == t.sched.count_grad_tot


def test_resume_refuses_checkpoint_with_foreign_optimizer_shards(workdir):
    """Shards written by another world size (or a missing shard of this rank) must be an error, not a silent cold start of this
    rank's Adam state (ranks would then disagree on bias correction, LR and the stop round and hang at the round barrier)."""
    import os
    import pytest
    a = dict(save=True, save_optimizer=True, nb_steps_tot=6)
    t = make("acco", **a)
    t.train()
    ckdir = workdir / "checkpoints"
    os.rename(ckdir / "job42_model_optim_rank0of1.pt", ckdir / "job42_model_optim_rank0of2.pt")
    with pytest.raises(FileNotFoundError):
        make("acco", resume_from=str(ckdir / "job42_model.pt"), **a)


def test_eval_and_checkpoint_tail_sees_committed_weights_only(workdir):
    """The periodic tail (eval / checkpoint) runs between `_complete_round` and `_launch_round`: nothing is in flight, the model is
    bound to the buffer the finished round wrote, and under ACCO only *real* rounds (committed weights) are evaluated / saved."""
    seen = []
    t = make("acco", nb_steps_tot=16, eval=True, eval_step=0, save=True, save_interval_s=0.0)
    orig_eval, orig_save = t.eval_loop, t.save_checkpoint

    def spy_eval():
        seen.append(("eval", t._inflight is None, t.arena.live, t.sched.round, t.sched.count_com))
        return orig_eval()

    def spy_save(path):
        seen.append(("save", t._inflight is None, t.arena.live, t.sched.round, t.sched.count_com))
        return orig_save(path)

    t.eval_loop, t.save_checkpoint = spy_eval, spy_save
    t.eval_dataset = t.train_dataset
    t.eval_dataloader = t.get_eval_dataloader()
    t.train()
    periodic = [s for s in seen if s[3] < 16]
    assert any(k == "eval" for k, *_ in periodic) and any(k == "save" for k, *_ in periodic)
    for kind, quiescent, live, rnd, ncom in seen:
        assert quiescent                                     # no communication round in flight
        assert live == rnd % 2                               # bound to the buffer the last finished round wrote
    # ACCO: tails happen after real rounds only -> an even number of completed rounds
    assert all(ncom % 2 == 0 for _, _, _, _, ncom in periodic), periodic


def test_label_smoothing_path(workdir):
    ds = synthetic_sft_dataset(60, 10, 96, 16, seed=1)
    tok = ByteTokenizer(); tok.pad_token_id = 95

    class Logits(torch.nn.Module):          # HF-style model returning logits under key "logits"
        def __init__(self):
            super().__init__()
            self.m = tiny_model()

        def forward(self, input_ids=None, labels=None, attention_mask=None, **kw):
            out = self.m(input_ids=input_ids)
            return {"logits": out.logits}

    t = DecoupledTrainer(model=Logits(), tokenizer=tok, train_dataset=ds,
                         args=base_args(const_len_batch=False, label_smoothing_factor=0.1, nb_steps_tot=4), log=LOG, env=DistEnv())
    t.train()
    assert torch.isfinite(t.loss_host).all()


def test_flat_accessors(workdir):
    t = make("acco")
    w = t.get_weights().clone()
    t.set_weights(w * 0 + 1)
    assert all(torch.all(p == 1) for p in t.model.parameters())
    t.set_grads(torch.full_like(t.get_grads(), 2.0))
    assert all(torch.all(p.grad == 2) for p in t.model.parameters())
    assert t.len_params == t.arena.numel and t.size_slice >= t.size_local_slice


class _DeferredRound:
    """Stand-in for the CUDA completion event of a round: the round 'finishes' only after `polls` queries
    (or when somebody blocks on it) - lets the CPU suite exercise the accumulate-while-communicating branch."""

    def __init__(self, polls, run):
        self.polls, self.run, self.ran = polls, run, False

    def _finish(self):
        if not self.ran:
            self.ran = True
            self.run()

    def query(self):
        if self.polls > 0:
            self.polls -= 1
            return False
        self._finish()
        return True

    def synchronize(self):
        self._finish()


def _make_async(t, polls_for_round):
    """Patch a CPU trainer so that round r needs `polls_for_round(r)` event polls before it completes."""
    from acco_b200.trainer import _InFlight

    def launch():
        plan = t.sched.next_plan()
        lr = t.lr_schedule.lr_at(t.sched)
        count = t._local_count
        t.round_history.append((plan.index, plan.kind, int(count)))
        evt = _DeferredRound(polls_for_round(plan.index), lambda: t.backend.launch_round(plan, lr, count))
        t._inflight = _InFlight(plan, evt, count)
        t._local_count = 0
    t._launch_round = launch


def test_accumulate_while_communicating_dynamic_counts(workdir):
    """Slow rounds (the event is polled at micro-batch boundaries, trainer_decoupled.py:497): the compute side keeps
    accumulating, the counts follow, and every committed update is still the mean over exactly the micro-batches it saw."""
    class Lin(torch.nn.Module):        # gradient independent of the weights -> the expected update is easy to state
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(6))
            self.k = 0

        def forward(self, input_ids=None, labels=None, **kw):
            self.k += 1
            return ((self.w * float(self.k)).sum(),)       # grad of micro-batch k is k * ones

    t = make("acco", model=Lin(), nb_steps_tot=10 ** 6, learning_rate=0.1, weight_decay=0.0, scheduler_name="constant",
             adam_beta1=0.0, adam_beta2=0.0)          # beta=0: the update is -lr * g/|g| = -lr * sign(mean grad) ... keep it simple
    _make_async(t, lambda r: 2 if r >= 0 else 0)       # every round needs 2 extra polls -> 3 micro-batches per phase
    flips = 0
    steps = 0
    while flips < 5:
        flipped = t.step()
        steps += 1
        flips += int(flipped)
    t._drain()
    counts = [c for _, _, c in t.round_history]
    # priming phase: 1 micro-batch; afterwards each phase runs until the in-flight round has been polled 3 times
    assert counts[0] == 1 and all(c == 3 for c in counts[1:]), counts
    # committed gradient count: real rounds (odd) add stash + current
    real = [i for i, (_, kind, _) in enumerate(t.round_history) if kind == "real"]
    expected_total = sum(counts[i - 1] + counts[i] for i in real if i < len(counts) and t.sched.count_com > i)
    assert t.sched.count_grad_tot == expected_total
    assert t.sharded_optimizer.step == sum(1 for i in real if t.sched.count_com > i)
    assert steps > flips                               # some step() calls only accumulated (no flip)


def test_profile_helper_writes_trace(workdir):
    t = make("acco", nb_steps_tot=10 ** 6)
    trace = t.profile(steps=2, warmup=1)
    assert os.path.isfile(trace) and os.path.getsize(trace) > 100
    assert os.path.isfile(os.path.join(os.path.dirname(trace), "ops_rank0.txt"))


@pytest.mark.parametrize("method", ["acco", "ddp"])
def test_hf_model_object_trains_through_the_trainer(workdir, method):
    """The reference hands `AutoModelForCausalLM.from_pretrained(...)` straight to DecoupledTrainer (`main.py:33-35`): any HF causal
    LM module must train through the generic path - its parameters are re-pointed into the flat arena (both theta buffers), the
    gradients accumulate in the arena, and the loss goes down."""
    transformers = pytest.importorskip("transformers")
    torch.manual_seed(0)
    hf = transformers.LlamaForCausalLM(transformers.LlamaConfig(
        vocab_size=96, hidden_size=32, intermediate_size=48, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
        max_position_embeddings=32, tie_word_embeddings=True, attn_implementation="eager"))
    ds = synthetic_pretrain_dataset(300, 30, 96, 16, seed=7)
    t = DecoupledTrainer(model=hf, train_dataset=ds, args=base_args(method_name=method, nb_steps_tot=40, learning_rate=1e-2, batch_size=4),
                         log=LOG, env=DistEnv(id_run="hf"))
    # every HF parameter (tied embedding counted once) lives in the arena
    assert t.len_params == sum(p.numel() for p in hf.parameters())
    losses = []
    while not t.finished():
        t.step()
        losses.append(float(t.loss_host))
    t._drain()
    assert all(l == l for l in losses) and sum(losses[-4:]) / 4 < sum(losses[:4]) / 4 - 0.05, losses
    live = t.arena.theta[t.arena.live]
    p0 = next(hf.parameters())
    assert p0.data_ptr() >= live.data_ptr() and p0.data_ptr() < live.data_ptr() + live.numel() * live.element_size()
    assert "model.embed_tokens.weight" in t.model.state_dict()         # checkpoint keys are the HF module's own


@pytest.mark.parametrize("method", ["acco", "dpu", "ddp"])
def test_debug_poison_mode_changes_nothing_when_the_protocol_is_right(workdir, method):
    """`debug_poison`: the parameter buffer a round is about to rewrite is NaN-filled first.  With a correct schedule compute never
    reads it while the round is in flight, so the run is bit-identical to the normal one and the loss stays finite; a wrong flip would
    surface as NaN immediately (race detector of SURVEY section 5)."""
    a = make(method, nb_steps_tot=12)
    a.train()
    b = make(method, nb_steps_tot=12, debug_poison=True)
    b.train()
    assert torch.isfinite(b.loss_host).all() and torch.isfinite(b.params).all()
    assert torch.equal(a.params, b.params)


def test_debug_poison_catches_a_wrong_buffer_binding(workdir):
    """Break the protocol on purpose: bind compute to the buffer the in-flight round is rewriting -> the host assertion fires."""
    t = make("acco", nb_steps_tot=12, debug_poison=True)
    t._begin_run()
    t.step()                                   # primes: round 0 launched (CPU backend: completes synchronously but stays "in flight")
    assert t._inflight is not None
    wrong = {"theta": t._inflight.plan.write_theta, "acc": t._inflight.plan.read_acc}
    t.sched.compute_buffers = lambda round_in_flight: wrong
    with pytest.raises(AssertionError):
        t._bind_compute_buffers()


def test_resume_auto_picks_the_latest_complete_checkpoint_and_limit_prunes(workdir):
    """`resume_from=auto`: newest checkpoint under ./checkpoints with a complete shard set (none -> fresh start);
    `save_total_limit` keeps only the newest periodic checkpoints."""
    a = dict(save=True, save_optimizer=True, nb_steps_tot=12, save_interval_s=0.0, save_total_limit=2)
    fresh = make("acco", resume_from="auto", **a)                      # nothing to resume from
    assert fresh.sched.count_grad_tot == 0
    fresh.train()
    files = sorted(os.listdir(workdir / "checkpoints"))
    periodic = [f for f in files if f.startswith("job42_model_") and "optim" not in f]
    assert len(periodic) == 2, files                                   # older periodic checkpoints were pruned (shards included)
    assert sum("optim" in f for f in files) == 3, files                # 2 periodic + the final one
    t2 = make("acco", resume_from="latest", **a)
    assert t2.sched.count_grad_tot == fresh.sched.count_grad_tot > 0 and t2.sharded_optimizer.step == fresh.sharded_optimizer.step
    torch.testing.assert_close(t2.params, fresh.params)


def test_resume_continues_the_data_stream(workdir):
    """The optimizer shard records how many batches this rank has consumed; a resumed run fast-forwards its loader (same seed, same
    epoch permutations) instead of replaying the data from the start."""
    a = dict(save=True, save_optimizer=True, nb_steps_tot=27, batch_size=4, seed=3)
    ds = synthetic_pretrain_dataset(10, 30, 96, 16, seed=3)       # small: the run crosses an epoch boundary
    t = make("acco", ds=ds, **a)
    t.train()
    st = torch.load(workdir / "checkpoints" / "job42_model_optim_rank0of1.pt", weights_only=False)
    consumed = st["data_batches"]
    assert consumed == t.micro_batches > len(t.train_dataloader)  # more than one epoch
    # what an uninterrupted run would read next
    ref = make("acco", ds=ds, **a)
    stream = []
    for _ in range(5):
        for idx in ref.train_dataloader.index_batches():
            stream.append(idx.tolist())
    t2 = make("acco", ds=ds, resume_from="auto", **a)
    nxt = next(iter(t2.train_dataloader.index_batches())).tolist()
    assert nxt == stream[consumed] and nxt != stream[0]


def test_reference_parity_ddp_mode_fp32_weights_with_bf16_autocast(workdir):
    """`run_baseline_ddp=True, ddp_weights_dtype=fp32, use_mixed_precision=True` = the reference's DDP baseline (fp32 weights, bf16
    autocast, `trainer_base.py:164-169`): forward runs under autocast, backward outside of it - LinearFn must cope with the bf16
    upstream gradient meeting fp32 saved tensors (advisor finding, round 1)."""
    t = make("ddp", run_baseline_ddp=True, ddp_weights_dtype="fp32", use_mixed_precision=True, nb_steps_tot=20, learning_rate=5e-3, batch_size=4)
    assert t.autocast and t.param_dtype == torch.float32 and t.dtype == torch.bfloat16
    losses = []
    while not t.finished():
        t.step()
        losses.append(float(t.loss_host))
    assert all(l == l for l in losses) and sum(losses[-4:]) < sum(losses[:4])
    assert t.params.dtype == torch.float32


def test_bf16_weights_mixed_precision_on_cpu(workdir):
    """`use_mixed_precision=True` on the sharded path: bf16 weights / gradients / accumulators, fp32 master shard."""
    t = make("acco", use_mixed_precision=True, nb_steps_tot=24, learning_rate=5e-3, batch_size=4)
    assert t.param_dtype == torch.bfloat16 and t.params.dtype == torch.bfloat16 and t.sharded_optimizer.master.dtype == torch.float32
    t.train()
    assert torch.isfinite(t.params.float()).all() and float(t.loss_host) == float(t.loss_host)


def test_grad_count_files_and_bounded_eval(workdir):
    """`save_grad_counts` (the reference's unused `save_grad_acc`, `utils/logs_utils.py:248`) writes one line of per-round
    micro-batch counts per rank; `max_eval_batches` bounds the eval pass; `eval_all_ranks` is a no-op switch on one rank."""
    ds = synthetic_pretrain_dataset(200, 30, 96, 16, seed=3)
    ev = synthetic_pretrain_dataset(80, 30, 96, 16, seed=4)
    t = DecoupledTrainer(model=tiny_model(), train_dataset=ds, eval_dataset=ev, log=LOG, env=DistEnv(id_run="job42"),
                         args=base_args(save_grad_counts=True, save_com_logs=True, eval=True, eval_step=2, max_eval_batches=2, eval_all_ranks=True, nb_steps_tot=12))
    calls = []
    orig = t._forward_loss
    t._forward_loss = lambda model, inputs: (calls.append(model.training), orig(model, inputs))[1]
    t.train()
    evals = [c for c in calls if not c]
    assert evals and len(evals) % 2 == 0                      # every eval pass stopped after exactly 2 batches
    assert open(workdir / "com_logs" / "job42_0.txt").read().startswith("0 rounds : [")
    txt = open(workdir / "grad_counts" / "job42_0.txt").read()
    assert txt.startswith("0 # grad acc : [") and "kinds" in txt
    n_rounds = len(t.round_history)
    assert txt.count(",") >= n_rounds - 1


def test_real_hf_datasets_objects_through_the_trainer(workdir):
    """The reference hands `datasets.Dataset` objects to the trainer (`main.py:49-50`, `trainer_base.py:100-124,193-200`:
    `.shard`, `.map(num_proc=...)`, `.column_names`): raw text with const-len packing, raw text pad-collated (SFT), and a
    pre-tokenised `input_ids` column."""
    datasets = pytest.importorskip("datasets")
    import numpy as np
    rng = np.random.default_rng(0)
    texts = ["".join(chr(97 + int(c)) for c in rng.integers(0, 26, size=int(rng.integers(20, 200)))) for _ in range(200)]
    ds = datasets.Dataset.from_dict({"text": texts}).train_test_split(0.05, seed=42)
    tok = ByteTokenizer()
    tok.pad_token_id = tok.eos_token_id
    common = dict(model=None, tokenizer=tok, train_dataset=ds["train"], eval_dataset=ds["test"], text_column_name="text", log=LOG)
    t = DecoupledTrainer(**{**common, "model": tiny_model(vocab=257)}, env=DistEnv(id_run="hf1"),
                         args=base_args(nb_steps_tot=8, max_length=32, eval=True, eval_step=4))
    assert t.train_dataset.column_names == ["input_ids"] and all(len(r) == 32 for r in t.train_dataset["input_ids"][:5])
    assert t.train()["count_grad_tot"] >= 8
    t2 = DecoupledTrainer(**{**common, "model": tiny_model(vocab=257)}, env=DistEnv(id_run="hf2"),
                          args=base_args(nb_steps_tot=8, max_length=32, const_len_batch=False, eval=True, eval_step=4))
    assert t2.train()["count_grad_tot"] >= 8
    ids = datasets.Dataset.from_dict({"input_ids": [list(map(int, rng.integers(0, 96, size=16))) for _ in range(120)]})
    t3 = DecoupledTrainer(model=tiny_model(), train_dataset=ids, args=base_args(nb_steps_tot=8), log=LOG, env=DistEnv(id_run="hf3"))
    assert t3.train()["count_grad_tot"] >= 8


@pytest.mark.parametrize("kind", ["dict", "SimpleNamespace", "argparse"])
def test_args_may_be_any_mapping_or_namespace(workdir, kind):
    """`args` is attribute-accessed in the reference (a Hydra DictConfig there, `main.py:60`); any mapping / namespace works here,
    missing keys fall back to the defaults of `config/train/*.yaml`."""
    import argparse
    raw = dict(base_args(nb_steps_tot=6))
    args = {"dict": dict(raw), "SimpleNamespace": types.SimpleNamespace(**raw), "argparse": argparse.Namespace(**raw)}[kind]
    t = DecoupledTrainer(model=tiny_model(), train_dataset=synthetic_pretrain_dataset(200, 30, 96, 16, seed=3), args=args, log=LOG,
                         env=DistEnv(id_run="ns"))
    assert t.train()["count_grad_tot"] >= 6


def test_public_accessors_of_the_reference_api(workdir):
    """`get_weights / set_weights / get_grads / set_grads` (`trainer_base.py:284-331`: flat vectors aliasing the model's
    parameters / gradients), `get_train_dataloader / get_eval_dataloader`, `warmup_steps`, `eval_loop` (SURVEY 2.9)."""
    ev = synthetic_pretrain_dataset(60, 30, 96, 16, seed=4)
    t = DecoupledTrainer(model=tiny_model(), train_dataset=synthetic_pretrain_dataset(200, 30, 96, 16, seed=3), eval_dataset=ev,
                         args=base_args(method_name="ddp", nb_steps_tot=6), log=LOG, env=DistEnv(id_run="api"))
    w = t.get_weights()
    assert w.dim() == 1 and w.numel() == sum(p.numel() for p in t.model.parameters())
    first = next(t.model.parameters())
    assert first.data_ptr() == w.data_ptr()                         # parameters are views of the flat vector
    t.set_weights(torch.zeros_like(w))
    assert float(first.abs().sum()) == 0.0
    t.set_weights(torch.full_like(w, 0.01))
    assert float(first.flatten()[0]) == pytest.approx(0.01)
    t.set_grads(torch.ones_like(t.get_grads()))
    assert float(first.grad.sum()) == first.numel()                 # gradients are views of the flat gradient vector
    tl, el = t.get_train_dataloader(), t.get_eval_dataloader()
    assert len(tl) == len(t.train_dataset) // t.batch_size and next(iter(el))["input_ids"].shape == (t.batch_size, 16)
    t._begin_run()
    t.warmup_steps(2)
    assert t.sched.count_com == 2 and t.sched.count_grad_tot == 2
    assert torch.isfinite(t.eval_loop())


def test_prepare_inputs_moves_nested_batches(workdir):
    t = make("ddp", nb_steps_tot=2)
    batch = {"input_ids": torch.ones(2, 4, dtype=torch.long), "extra": [torch.zeros(1), ("keep", 3)], "n": 7}
    out = t._prepare_inputs(batch)
    assert out["input_ids"].device == t.device and out["extra"][0].device == t.device and out["extra"][1] == ("keep", 3) and out["n"] == 7
    loss = t.compute_loss(t.model, {"input_ids": torch.randint(0, 96, (2, 8)), "labels": torch.randint(0, 96, (2, 8))})
    assert loss.dim() == 0 and torch.isfinite(loss)


def test_reference_attribute_names_are_readable(workdir):
    """Attributes user code reads off the reference trainer: sizes, ranks, optimizer shard, LR scheduler, counters, iterators."""
    t = make("acco", nb_steps_tot=8, scheduler_name="cosine", warmup=2)
    for name in ("rank", "local_rank", "world_size", "node_id", "n_nodes", "id_run", "batch_size", "nb_grad_tot", "len_params", "size_slice",
                 "size_local_slice", "params", "params_opt", "sharded_optimizer", "loss_static", "train_dataloader", "master_addr", "master_port"):
        assert getattr(t, name) is not None, name
    assert t.count_grad_local == 0 and t.count_grad_this_round == 0
    batch = next(t.train_iterator)
    assert batch["input_ids"].shape == (t.batch_size, 16)
    t.train()
    assert t.count_grad_this_round >= 1
    (lr,) = t.scheduler.get_last_lr()
    assert 0 < lr <= float(t.args.learning_rate)


def test_callbacks_fire_between_rounds_and_early_stopping_stops(workdir):
    from acco_b200 import EarlyStoppingCallback, TrainerCallback

    class Recorder(TrainerCallback):
        def __init__(self):
            self.events = []

        def on_train_begin(self, trainer):
            self.events.append("begin")

        def on_round_end(self, trainer, plan):
            assert trainer._inflight is None                      # between rounds: nothing in flight
            self.events.append(("round", plan.kind))

        def on_evaluate(self, trainer, eval_loss):
            self.events.append(("eval", round(eval_loss, 3)))

        def on_save(self, trainer, path):
            self.events.append(("save", os.path.basename(path)))

        def on_train_end(self, trainer, stats):
            self.events.append(("end", stats["count_grad_tot"]))

    ds = synthetic_pretrain_dataset(200, 30, 96, 16, seed=3)
    ev = synthetic_pretrain_dataset(60, 30, 96, 16, seed=4)
    t = DecoupledTrainer(model=tiny_model(), train_dataset=ds, eval_dataset=ev, log=LOG, env=DistEnv(id_run="cb"),
                         args=base_args(nb_steps_tot=12, eval=True, eval_step=3, save=True))
    rec = Recorder()
    t.add_callback(rec)
    t.train()
    kinds = [e[0] if isinstance(e, tuple) else e for e in rec.events]
    assert kinds[0] == "begin" and kinds[-1] == "end" and "eval" in kinds and ("save", "cb_model.pt") in rec.events
    assert all(k == "real" for tag, k in (e for e in rec.events if isinstance(e, tuple) and e[0] == "round"))    # ACCO: committed rounds only
    # early stopping: a learning rate of zero never improves the eval loss
    t2 = DecoupledTrainer(model=tiny_model(), train_dataset=ds, eval_dataset=ev, log=LOG, env=DistEnv(id_run="es"),
                          args=base_args(method_name="ddp", nb_steps_tot=10 ** 6, eval=True, eval_step=1, learning_rate=0.0))
    t2.add_callback(EarlyStoppingCallback(patience=2))
    stats = t2.train()
    assert stats["count_grad_tot"] < 50
