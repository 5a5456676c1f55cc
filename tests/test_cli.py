import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_main_cli_end_to_end(workdir):
    sys.path.insert(0, ROOT)
    import main as cli
    stats = cli.main(["train=acco", "model=tiny", "data=synthetic", "train.nb_steps_tot=6", "train.batch_size=2", "train.max_length=32",
                      "train.use_mixed_precision=False", "data.synthetic_docs=200", "data.synthetic_mean_len=40", "train.warmup=0",
                      "run_name=clitest", "train.save=True"])
    assert stats["count_grad_tot"] >= 6
    assert os.path.isdir(workdir / "tensorboard" / "clitest")
    assert any(f.endswith("_model.pt") for f in os.listdir(workdir / "checkpoints"))
    assert os.path.exists(workdir / "results.csv")


def test_sft_cli(workdir):
    import main as cli
    stats = cli.main(["train=acco-ft", "model=tiny", "data=alpaca", "train.nb_steps_tot=8", "train.max_length=32", "train.eval_step=2",
                      "train.use_mixed_precision=False", "data.synthetic_docs=120", "data.synthetic_mean_len=12"])
    assert stats["count_grad_tot"] >= 8


def test_shim_import():
    import trainer_decoupled as td
    import decoupled_trainer as dt
    import importlib.util
    # by file path: this repo's shim, whatever module another import may have registered as `trainer_base` in sys.modules
    spec = importlib.util.spec_from_file_location("trainer_base_shim", os.path.join(ROOT, "trainer_base.py"))
    tb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tb)
    from acco_b200 import DecoupledTrainer
    assert td.DecoupledTrainer is DecoupledTrainer is dt.DecoupledTrainer
    assert issubclass(DecoupledTrainer, tb.DecoupledTrainerBase)         # `trainer_base.DecoupledTrainerBase` of the reference
    for name in ("initialize_com", "prepare_data", "get_train_dataloader", "get_eval_dataloader", "get_weights", "set_weights", "get_grads", "set_grads",
                 "_prepare_input", "_prepare_inputs", "compute_loss"):
        assert callable(getattr(tb.DecoupledTrainerBase, name)), name


def test_dl_dataset_and_perplexity(workdir):
    import dl_dataset
    saved = dl_dataset.main(["model=tiny", "train.max_length=32", f"out={workdir}/tok", "num_proc=1", "data.synthetic_docs=50"])
    from acco_b200.data import load_from_disk
    tr = load_from_disk(saved["train"][0])
    assert tr.column_names == ["input_ids"] and all(len(r) == 32 for r in tr["input_ids"])
    import perplexity_eval
    res = perplexity_eval.main(["model=tiny", "n=6", "batch_size=4", "max_length=24"])
    assert len(res["perplexities"]) == 6 and all(p > 1 for p in res["perplexities"])


def test_perplexity_matches_manual():
    from acco_b200.data import ByteTokenizer
    from acco_b200.eval import compute_perplexity
    from acco_b200.models import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(0)
    m = LlamaForCausalLM(LlamaConfig(vocab_size=257, hidden_size=32, intermediate_size=48, num_hidden_layers=1, num_attention_heads=2,
                                     max_position_embeddings=64, pad_vocab_multiple=8)).float()
    tok = ByteTokenizer()
    texts = ["hello world", "acco"]
    res = compute_perplexity(m, tok, texts, batch_size=2, add_start_token=True, max_length=32)
    ids = torch.tensor([[256] + list(b"acco")])
    lp = torch.log_softmax(m(input_ids=ids).logits[:, :-1].float(), -1).gather(-1, ids[:, 1:, None]).squeeze(-1)
    assert res["perplexities"][1] == pytest.approx(float(torch.exp(-lp.mean())), rel=1e-4)


def test_shim_step_primitives_drive_a_round(workdir):
    """`trainer_decoupled.{gradient_step, communication_step, update_buffers_step}` (the reference's free functions,
    `trainer_decoupled.py:18-126`) really run a micro-batch, a full round and the buffer flip on the trainer."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import trainer_decoupled as td
    from acco_b200.data import synthetic_pretrain_dataset
    from acco_b200.launch import DistEnv
    from helpers import LOG, base_args, tiny_model
    ds = synthetic_pretrain_dataset(200, 30, 96, 16, seed=7)
    t = td.DecoupledTrainer(model=tiny_model(), train_dataset=ds, args=base_args(method_name="ddp"), log=LOG, env=DistEnv(id_run="shim"))
    t._begin_run()
    td.update_buffers_step(t)
    before = t.params.clone()
    td.gradient_step(t)
    assert float(t.get_grads().abs().sum()) > 0 and t._local_count == 1
    plan = td.communication_step(t)
    assert plan.kind == "sync" and t.sched.count_com == 1 and t.sched.count_grad_tot == 1
    td.update_buffers_step(t)
    assert not torch.equal(t.params, before)                     # the model now reads the weights the round produced
    assert float(t.arena.acc[plan.read_acc].abs().sum()) == 0    # the consumed accumulator was cleared


@pytest.mark.parametrize("train,data", [("dpu", "synthetic"), ("ddp", "synthetic"), ("dpu-ft", "alpaca"), ("ddp-ft", "alpaca")])
def test_every_shipped_train_config_runs(workdir, train, data):
    """`config/train/{dpu,ddp,dpu-ft,ddp-ft}.yaml` through `main.py` (acco / acco-ft are covered above): warm-up rounds, eval
    cadence, pad-collated SFT batches, synchronous DDP."""
    import main as cli
    stats = cli.main([f"train={train}", "model=tiny", f"data={data}", "data.synthetic=true", "train.nb_steps_tot=16", "train.batch_size=2",
                      "train.max_length=32", "train.use_mixed_precision=False", "data.synthetic_docs=120", "data.synthetic_mean_len=20",
                      "train.warmup=0", "train.n_warmup_steps=2", "train.tensorboard=False", "train.save=False", "train.eval_step=4"])
    assert stats["count_grad_tot"] >= 16 and stats["backend"] == "gloo"


def test_reference_readme_snippet_runs(workdir):
    """The usage snippet of the reference's README (`/root/reference/README.md:88-110`: HF `LlamaForCausalLM`, a tokenizer, HF
    datasets, `from decoupled_trainer import DecoupledTrainer`, no `log` argument) works unchanged against this package."""
    transformers = pytest.importorskip("transformers")
    datasets = pytest.importorskip("datasets")
    import numpy as np
    from decoupled_trainer import DecoupledTrainer
    from acco_b200 import compose
    from acco_b200.data import ByteTokenizer
    model = transformers.LlamaForCausalLM(transformers.LlamaConfig(vocab_size=257, hidden_size=32, intermediate_size=64, num_hidden_layers=1,
                                                                  num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=64))
    tokenizer = ByteTokenizer()
    tokenizer.pad_token_id = tokenizer.eos_token_id
    rng = np.random.default_rng(0)
    texts = ["".join(chr(97 + int(c)) for c in rng.integers(0, 26, size=int(rng.integers(20, 200)))) for _ in range(120)]
    dataset = datasets.DatasetDict({"train": datasets.Dataset.from_dict({"text": texts}), "validation": datasets.Dataset.from_dict({"text": texts[:20]})})
    train_config = compose(overrides=["train=acco", "train.nb_steps_tot=8", "train.batch_size=2", "train.max_length=32", "train.use_mixed_precision=False",
                                      "train.tensorboard=False", "train.save=False", "train.warmup=0"]).train
    trainer = DecoupledTrainer(model=model, tokenizer=tokenizer, train_dataset=dataset["train"], eval_dataset=dataset["validation"],
                               text_column_name="text", args=train_config)
    assert trainer.train()["count_grad_tot"] >= 8


def test_perplexity_eval_of_an_hf_checkpoint_directory(tmp_path):
    """`perplexity_eval.py pretrained=<HF dir>`: the reference evaluates HF checkpoints (`perplexity_eval.py:13-30`)."""
    transformers = pytest.importorskip("transformers")
    torch.manual_seed(0)
    hf = transformers.LlamaForCausalLM(transformers.LlamaConfig(vocab_size=300, hidden_size=32, intermediate_size=64, num_hidden_layers=1,
                                                               num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=64))
    hf.save_pretrained(tmp_path / "ck")
    import perplexity_eval
    res = perplexity_eval.main([f"pretrained={tmp_path / 'ck'}", "n=4", "batch_size=2", "max_length=24"])
    assert len(res["perplexities"]) == 4 and all(p > 1 for p in res["perplexities"])


def test_hydra_style_run_directory(workdir):
    """Like Hydra (`config/config.yaml:10-12`): `outputs/<date>/<time>/.hydra/{config,overrides}.yaml` + `main.log`, no chdir."""
    import yaml
    import main as cli
    cli.main(["train=acco", "model=tiny", "data=synthetic", "train.nb_steps_tot=4", "train.batch_size=2", "train.max_length=32",
              "train.use_mixed_precision=False", "data.synthetic_docs=100", "data.synthetic_mean_len=40", "train.tensorboard=False", "train.save=False"])
    days = os.listdir(workdir / "outputs")
    assert len(days) == 1
    run = workdir / "outputs" / days[0] / os.listdir(workdir / "outputs" / days[0])[0]
    cfg = yaml.safe_load(open(run / ".hydra" / "config.yaml"))
    assert cfg["train"]["method_name"] == "acco" and cfg["train"]["nb_steps_tot"] == 4 and cfg["model"]["arch"] == "llama" and "hydra" not in cfg
    assert "train.nb_steps_tot=4" in yaml.safe_load(open(run / ".hydra" / "overrides.yaml"))
    assert (run / "main.log").exists() and os.path.exists(workdir / "results.csv")       # artefacts stay in the launch directory
