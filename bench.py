#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): training throughput in tokens/s, Llama-125M ACCO, bf16,
sharded AdamW, synthetic openwebtext-shaped const-len batches of 8 x 1024 tokens per GPU
(`config/train/acco.yaml` of the reference), weak scaling over 1/2/4/8 B200.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus 8 --steps 20 --warmup 5
    python bench.py --impl reference ...      # the unmodified reference trainer on the same config

A *step* is one scheduling iteration of the trainer's public ``step()``: ``n_grad_accumulation``
micro-batches per rank (forward + backward, gradients accumulated in the flat arena) plus - when the
previous round has finished, which is every step in steady state - one full communication round
(reduce-scatter, sharded AdamW, all-gather) overlapped with the next step's compute.  Nothing is
skipped: optimizer, both ACCO half-rounds, LR schedule and loss read-out all run inside the timed
region.  Throughput counts the micro-batches actually executed (summed over ranks) x 8 x 1024 tokens,
divided by the device-timed duration (CUDA events on the compute stream, barrier + synchronize on
both sides, MAX over ranks).

Two timed passes: ``value`` with inputs already resident on the device (isolates the GPU work), and
``e2e`` where every micro-batch's tokens come from pinned host memory (async H2D) and every step's
loss is read back to the host - both through ``DecoupledTrainer.step()``, the loop ``train()`` runs.
"""
from __future__ import annotations

import argparse
import json
import logging
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "tokens/sec (device-timed, max over ranks) Llama ACCO bf16 sharded-Adam, 8x1024 tokens per GPU per micro-batch"


class ClockSampler:
    """Samples `nvidia-smi` clocks / throttle reasons while the timed region runs (rank 0 only)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, n_gpus: int):
        self.n, self.proc, self.lines = n_gpus, None, []
        self.t_mark = None

    def mark(self):
        """Start of the timed region: samples that arrive before it (warm-up) are only used if the region is too short to be sampled
        (nvidia-smi needs ~1 s to start with 8 GPUs, the driver's default timed region is ~0.2 s)."""
        self.t_mark = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._read, daemon=True)
            self._t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            self._t.join(timeout=2)                 # the reader ends with the pipe's EOF; do not leave it to interpreter shutdown
        except Exception:
            pass
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines
        inside = [ln for (ts, ln) in lines if self.t_mark is None or ts >= self.t_mark]
        scope = "timed region"
        if len(inside) < self.n:                    # region shorter than one sampling period: fall back to the loaded warm-up samples
            inside, scope = [ln for (_, ln) in lines], "warm-up + timed region"
        self.scope = scope
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                if int(f[0]) >= self.n:
                    continue
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nme, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return None
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "power_w_max": max(power), "samples": len(sm),
                "reasons": sorted(reasons), "scope": getattr(self, "scope", "timed region")}


# BASELINE.json configurations beyond the headline one (config 2 = the default flags).  The reference arm honours them too.
PRESETS_BENCH = {
    "llama125m": dict(model="llama125m", batch=8, seq=1024, n_acc=1, method="acco"),              # config 2 (headline)
    "llama125m-b1": dict(model="llama125m", batch=1, seq=1024, n_acc=1, method="acco"),            # comm/compute ~ 1: overlap matters
    "llama125m-ddp": dict(model="llama125m", batch=8, seq=1024, n_acc=1, method="ddp"),            # config 5 (synchronous baseline)
    "llama125m-b1-ddp": dict(model="llama125m", batch=1, seq=1024, n_acc=1, method="ddp"),
    "llama1b-b1": dict(model="llama3-1b", batch=1, seq=1024, n_acc=1, method="acco"),                # comm ~ compute on a 1.2 B model
    "llama1b-b1-ddp": dict(model="llama3-1b", batch=1, seq=1024, n_acc=1, method="ddp"),
    "llama1b-nacc1": dict(model="llama3-1b", batch=4, seq=1024, n_acc=1, method="acco"),
    "llama1b-nacc8": dict(model="llama3-1b", batch=4, seq=1024, n_acc=8, method="acco"),           # config 3
    "llama1b-nacc1-ddp": dict(model="llama3-1b", batch=4, seq=1024, n_acc=1, method="ddp"),
}


def model_kwargs(name: str):
    from acco_b200.models import PRESETS
    arch, kw = PRESETS[name]
    assert arch == "llama", "the headline benchmark is a Llama config"
    kw = dict(kw)
    kw.setdefault("num_key_value_heads", kw["num_attention_heads"])
    return kw


DUMP_PARAM_SAMPLE = 1 << 22      # --dump-outputs: a larger parameter vector is sampled down to this many elements (16 MB of float32)


def dump_outputs(out_dir: str, trainer) -> None:
    """Write what ``trainer.step()`` hands its caller once the last timed step's round has landed, as float32 ``.npy`` files:
    ``loss`` (the last micro-batch's loss as read by the host) and ``params`` (the flat weight vector the model reads; above
    DUMP_PARAM_SAMPLE elements, the elements at a fixed sorted sample of indices drawn with seed 0).

    ACCO accumulates extra micro-batches while a round is still running, so how many ran depends on timing, and so do the inputs
    the last step saw.  ``micro_batches`` (this rank's, whole run) and ``count_grad_tot`` (committed gradients, all ranks) are
    written too, as float64: two dumps are comparable output for output only when these agree."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    params = trainer.params.detach()
    if params.numel() > DUMP_PARAM_SAMPLE:
        idx = torch.randint(params.numel(), (DUMP_PARAM_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        params = params[idx.to(params.device)]
    np.save(os.path.join(out_dir, "loss.npy"), trainer.loss_host.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "params.npy"), params.float().cpu().numpy())
    np.save(os.path.join(out_dir, "micro_batches.npy"), np.array([trainer.micro_batches], dtype=np.float64))
    np.save(os.path.join(out_dir, "count_grad_tot.npy"), np.array([trainer.sched.count_grad_tot], dtype=np.float64))


def run_ours(a) -> dict:
    import torch
    import torch.distributed as dist
    from acco_b200 import AttrDict, DecoupledTrainer, ops
    from acco_b200.data import TokenDataset
    from acco_b200.launch import discover_env, init_distributed
    from acco_b200.models import preset

    # the benchmark must produce a number even on a box whose symmetric-memory bring-up fails: allow the NCCL library path there
    # (the JSON line reports the backend that actually ran in config.comm_backend)
    os.environ.setdefault("ACCO_ALLOW_NCCL_FALLBACK", "1")
    env = init_distributed(discover_env())
    rank, world = env.rank, env.world_size
    dev = torch.device("cuda", env.local_rank)
    kw = model_kwargs(a.model)
    torch.manual_seed(1234)
    model = preset(a.model, device=dev, dtype=torch.bfloat16)   # construct + initialise on the GPU
    g = torch.Generator().manual_seed(7)
    rows = 64 * a.batch * world
    ds = TokenDataset({"input_ids": torch.randint(0, kw["vocab_size"], (rows, a.seq), generator=g, dtype=torch.long)})
    targs = AttrDict(   # `config/train/acco.yaml` values of the reference
        method_name=a.method, run_baseline_ddp=(a.method == "ddp"), batch_size=a.batch, n_grad_accumulation=a.n_acc,
        max_length=a.seq, learning_rate=6e-4, weight_decay=0.1, adam_beta1=0.9, adam_beta2=0.95, scheduler_name="cosine",
        warmup=1000, nb_steps_tot=10 ** 12, n_warmup_steps=0, use_mixed_precision=True, const_len_batch=True, eval=False,
        save=False, tensorboard=False, comm_backend=a.backend, cuda_graphs=not a.no_graphs, seed=1234, log_every=10 ** 9,
        fused_ag_gemm=bool(a.fused_ag), run_expe_slow=a.slow_ms > 0, slow_ranks=[a.slow_rank], slow_factor_ms=a.slow_ms)
    log = logging.getLogger("bench")
    log.setLevel(logging.WARNING)
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="acco_bench_")
    os.chdir(tmp)
    try:
        trainer = DecoupledTrainer(model=model, train_dataset=ds, args=targs, log=log, run_name="bench")

        def timed(n_steps: int):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            m0, l0 = trainer.micro_batches, ops.total_launches()
            h0 = trainer._feed().h2d_bytes
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            if a.slow_ms > 0 or a.by_count:
                # heterogeneous ranks: run until the GLOBAL committed-gradient counter has advanced by n_steps*world*n_acc, like
                # train() does - every rank leaves after the same round, and fast ranks are free to accumulate extra micro-batches
                target = trainer.sched.count_grad_tot + n_steps * world * a.n_acc
                while trainer.sched.count_grad_tot < target:
                    trainer.step()
            else:
                # a "step" = one round flip (n_acc micro-batches per rank + one overlapped round): with the gated round barrier a
                # rank that polls a moment before its peers arrive accumulates one more micro-batch instead of flipping, so the loop
                # counts FLIPS - every rank launches exactly n_steps rounds (no rank can leave a peer's round waiting)
                flips = 0
                while flips < n_steps:
                    flips += 1 if trainer.step() else 0
            e1.record()
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            if world > 1:
                dist.barrier()
            ms = e0.elapsed_time(e1)
            t = torch.tensor([ms, wall, float(trainer.micro_batches - m0), float(ops.total_launches() - l0),
                              float(trainer._feed().h2d_bytes - h0)], dtype=torch.float64, device=dev)
            tmax, tsum = t.clone(), t.clone()
            if world > 1:
                dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            return {"ms": float(tmax[0]), "wall_ms": float(tmax[1]), "micro": float(tsum[2]), "launches": float(t[3]),
                    "h2d": float(t[4])}

        # -------- pass 1: device-resident inputs (headline `value`)
        pool = [{"input_ids": torch.randint(0, kw["vocab_size"], (a.batch, a.seq), device=dev)} for _ in range(8)]
        it = [0]

        def from_pool():
            it[0] += 1
            return pool[it[0] % len(pool)]
        trainer.input_override = from_pool
        sampler = ClockSampler(world) if rank == 0 else None
        if sampler:
            sampler.start()
        flips = 0
        while flips < max(a.warmup, 3):
            flips += 1 if trainer.step() else 0
        if sampler:
            sampler.mark()
        r_dev = timed(a.steps)
        clocks = sampler.stop() if sampler else None
        # -------- pass 2: end to end (pinned host -> device per micro-batch, loss -> host per step)
        trainer.input_override = None
        flips = 0
        while flips < 3:
            flips += 1 if trainer.step() else 0
        r_e2e = timed(a.steps)
        overlap = trainer.overlap.summary()
        backend = trainer.backend.name
        loss = float(trainer.loss_host.item())
        n_params = trainer.len_params
        trainer._drain()
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, trainer)
    finally:
        os.chdir(cwd)
    tok = a.batch * a.seq
    value = r_dev["micro"] * tok / (r_dev["ms"] / 1e3)
    e2e = r_e2e["micro"] * tok / (r_e2e["ms"] / 1e3)
    from acco_b200.models import LlamaConfig
    flops_tok = LlamaConfig.from_dict(kw).flops_per_token(a.seq)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    mfu = value / world * flops_tok / (peaks.get("bf16_tflops_sustained", 1400.0) * 1e12)
    return {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": r_dev["ms"] / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic (uniform random token ids, random-init weights)", "impl": "acco_b200",
        "config": {"model": f"{a.model} ({n_params} params incl. LM-head row padding to a multiple of 128)", "global_batch": a.batch * a.n_acc * world,
                   "micro_batch_per_gpu": a.batch, "seq_len": a.seq, "n_grad_accumulation": a.n_acc, "method": a.method,
                   "parallelism": f"dp{world}+zero1", "comm_backend": backend, "cuda_graphs": not a.no_graphs, "fused_ag_gemm": bool(a.fused_ag), "slow_rank_ms": a.slow_ms,
                   "step": "one trainer.step(): n_acc micro-batches/rank + one overlapped RS+AdamW+AG round",
                   "l2": "per-step working set (250 MB weights x2 + >1 GB activations) exceeds the 126 MB L2; no explicit flush",
                   "micro_batches_timed": r_dev["micro"]},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "tokens/s", "ms_per_step": r_e2e["ms"] / a.steps, "wall_ms_per_step": r_e2e["wall_ms"] / a.steps,
                "h2d_bytes_per_step": r_e2e["h2d"] / a.steps, "d2h_bytes_per_step": 4 + 4,
                "api": "DecoupledTrainer.step() (the loop body of .train())"},
        "gpu_launches": int(r_dev["launches"]),
        "launch_breakdown": ops.launch_counts(),
        "mfu_vs_measured_sustained_bf16": mfu,
        "comm_ms_per_round": overlap["comm_ms_mean"], "exposed_comm_ms_per_round": overlap["exposed_ms_mean"],
        "final_loss": loss,
    }


def run_reference_arm(a) -> dict:
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    from run_reference import reference_available, run_reference
    why = reference_available()
    if why:
        return {"impl": "reference", "unavailable": why}
    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    sampler = ClockSampler(world) if rank == 0 else None
    if sampler:
        sampler.start()
    try:
        r = run_reference(a.steps, max(a.warmup, 3), model_kwargs(a.model), a.batch, a.seq, a.n_acc)
    except Exception as e:
        if sampler:
            sampler.stop()
        return {"impl": "reference", "unavailable": f"{type(e).__name__}: {str(e)[:300]}"}
    clocks = sampler.stop() if sampler else None
    value = r["tokens"] / (r["ms_total"] / 1e3)
    return {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": r["ms_total"] / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic (uniform random token ids, random-init weights)", "impl": "reference",
        "config": {"model": f"{a.model} (HF LlamaForCausalLM)", "global_batch": a.batch * a.n_acc * world, "micro_batch_per_gpu": a.batch,
                   "seq_len": a.seq, "n_grad_accumulation": a.n_acc, "method": "acco", "parallelism": f"dp{world}+zero1",
                   "comm_backend": "nccl (reference trainer_decoupled)", "micro_batches_timed": r["micro_batches"],
                   "note": "clock sample spans construction + warm-up + timed call"},
        "clocks": clocks,
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": r["h2d_bytes_per_step"], "d2h_bytes_per_step": r["d2h_bytes_per_step"],
                "api": "reference DecoupledTrainer.train() (always end-to-end: DataLoader -> .to(device) -> loss)"},
        "gpu_launches": 0, "final_loss": r["loss"],
    }


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20, help="timed steps (round flips) in each of the two timed passes")
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--model", default="llama125m")
    p.add_argument("--batch", type=int, default=8)
    p.add_argument("--seq", type=int, default=1024)
    p.add_argument("--n-acc", dest="n_acc", type=int, default=1)
    p.add_argument("--method", default="acco", choices=["acco", "dpu", "ddp"])
    p.add_argument("--backend", default="auto")
    p.add_argument("--no-graphs", action="store_true")
    p.add_argument("--fused-ag", dest="fused_ag", action="store_true",
                   help="pull remote weight row-blocks inside the first forward GEMM (KERNEL B) instead of pushing them in the round kernel")
    p.add_argument("--by-count", dest="by_count", action="store_true", help="time until the global gradient counter advanced by steps*world*n_acc")
    p.add_argument("--slow-rank", dest="slow_rank", type=int, default=1, help="rank slowed down when --slow-ms > 0 (heterogeneity experiment)")
    p.add_argument("--slow-ms", dest="slow_ms", type=float, default=0.0, help="extra GPU milliseconds per micro-batch on the slow rank")
    p.add_argument("--preset", default=None, choices=sorted(PRESETS_BENCH),
                   help="named BASELINE.json configurations (override --model/--batch/--seq/--n-acc/--method)")
    p.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                   help="after the timed steps, write the last step's loss and weights (sampled) and the micro-batch / gradient "
                        "counts that decide whether two dumps are comparable to DIR/*.npy (rank 0)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs:
        if a.impl == "reference":
            p.error("--dump-outputs applies to --impl ours")
        a.dump_outputs = os.path.abspath(a.dump_outputs)    # run_ours() works in a temporary directory
    if a.preset:
        for k, v in PRESETS_BENCH[a.preset].items():
            setattr(a, k, v)
    world = int(os.environ.get("WORLD_SIZE", 1))
    if a.gpus != world and world == 1 and a.gpus > 1:
        # convenience: re-launch ourselves under torchrun when called bare with --gpus N
        from acco_b200.launch import free_port
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(free_port()), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    out = run_reference_arm(a) if a.impl == "reference" else run_ours(a)
    if int(os.environ.get("RANK", 0)) == 0:
        print(json.dumps(out), flush=True)
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
