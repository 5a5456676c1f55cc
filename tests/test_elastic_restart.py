"""Failure drill, end to end on CPU (gloo): a rank dies mid-run -> its peer fails in the next collective -> torchrun restarts the
worker group -> `resume_from=auto` picks up the newest complete checkpoint -> the job finishes.  (The reference hangs forever when a
rank dies: no timeout, no restart, no resume - SURVEY section 5.)"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def clean_env(**extra):
    """Environment of a child job: nothing of THIS process's rendezvous (earlier in-process tests leave MASTER_PORT etc. behind,
    and that port is held by this very process)."""
    drop = ("MASTER_ADDR", "MASTER_PORT", "RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "GROUP_RANK")
    env = {k: v for k, v in os.environ.items() if k not in drop and not k.startswith(("SLURM_", "TORCHELASTIC_"))}
    env.update(OMP_NUM_THREADS="2", PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES="", **extra)     # CPU ranks even where a GPU is present
    return env


def test_rank_failure_restart_and_auto_resume(tmp_path):
    from acco_b200.launch import free_port
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--max-restarts=1", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), os.path.join(ROOT, "main.py"), "train=acco", "model=tiny", "data=synthetic", "train.nb_steps_tot=60",
           "train.batch_size=2", "train.max_length=32", "train.use_mixed_precision=False", "data.synthetic_docs=200", "data.synthetic_mean_len=40",
           "train.warmup=0", "train.tensorboard=False", "train.save=True", "train.save_optimizer=True", "train.save_interval_s=0",
           "train.save_total_limit=2", "train.resume_from=auto", "train.fault_inject=1@24", "train.log_every=1000000"]
    env = clean_env(ACCO_RUN_ID="drill")
    p = subprocess.run(cmd, cwd=tmp_path, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=240)
    out = p.stdout
    assert p.returncode == 0, out[-4000:]
    assert (tmp_path / "fault_injected.marker").exists()
    assert "fault_inject: rank 1 exits now" in out
    # second incarnation: resumed from a checkpoint written before the crash, with the Adam state and the counters
    assert "resume_from=auto: resuming from" in out and "no checkpoint found, starting fresh" in out
    files = os.listdir(tmp_path / "checkpoints")
    assert "drill_model.pt" in files and "drill_model_optim_rank0of2.pt" in files and "drill_model_optim_rank1of2.pt" in files
    import torch
    st = torch.load(tmp_path / "checkpoints" / "drill_model_optim_rank0of2.pt", weights_only=False)
    assert st["scheduler"]["count_grad_tot"] >= 60 and st["optimizer"]["step"] > 0


def test_sigterm_checkpoints_and_stops_then_auto_resume_continues(tmp_path):
    """`train.preempt_save=True`: SIGTERM (Slurm pre-emption / end of allocation) -> a complete checkpoint at the next committed
    round, clean exit 0; the requeued job (`resume_from=auto`) continues from it."""
    import signal
    import time
    import torch
    common = [sys.executable, os.path.join(ROOT, "main.py"), "train=acco", "model=tiny", "data=synthetic", "train.batch_size=2", "train.max_length=32",
              "train.use_mixed_precision=False", "data.synthetic_docs=200", "data.synthetic_mean_len=40", "train.warmup=0", "train.tensorboard=False",
              "train.save=True", "train.save_optimizer=True", "train.save_interval_s=100000", "train.preempt_save=True", "train.resume_from=auto",
              "train.log_every=50"]
    env = clean_env(ACCO_RUN_ID="preempt")
    p = subprocess.Popen(common + ["train.nb_steps_tot=100000000"], cwd=tmp_path, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    lines = []
    deadline = time.time() + 120
    while time.time() < deadline:                      # wait until training is under way (first progress line)
        line = p.stdout.readline()
        if not line:
            break
        lines.append(line)
        if "grad" in line.lower() and "loss" in line.lower():
            break
    p.send_signal(signal.SIGTERM)
    out, _ = p.communicate(timeout=120)
    out = "".join(lines) + out
    assert p.returncode == 0, out[-3000:]
    assert "pre-empted: checkpoint" in out
    files = sorted(os.listdir(tmp_path / "checkpoints"))
    models = [f for f in files if f.startswith("preempt_model_") and "optim" not in f]
    assert len(models) == 1 and f"{models[0][:-3]}_optim_rank0of1.pt" in files, files
    st = torch.load(tmp_path / "checkpoints" / f"{models[0][:-3]}_optim_rank0of1.pt", weights_only=False)
    done = int(st["scheduler"]["count_grad_tot"])
    assert done > 0 and str(done) in models[0]
    # requeue: a short run that only needs a few more gradients
    r = subprocess.run(common + [f"train.nb_steps_tot={done + 8}"], cwd=tmp_path, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=240)
    assert r.returncode == 0, r.stdout[-3000:]
    assert f"resuming from {tmp_path / 'checkpoints' / models[0]}" in r.stdout
    assert "preempt_model.pt" in os.listdir(tmp_path / "checkpoints")          # the resumed run finished normally
