"""CPU: the UNMODIFIED reference script training/train_maskgit_imagenet.py runs for two optimizer steps against the drop-in
``muse`` package, with the C-ABI kernels replaced by shape/dtype-checking stand-ins (the numerics are the GPU twin's job,
tests/test_train_script_gpu.py).  What this pins is the host-side surface the script relies on: constructor kwargs from
the yaml, ``config.mask_token_id``, ``requires_grad_``, ``enable_xformers_memory_efficient_attention``, the forward
keywords, ``parameters()`` into AdamW, the prepare / accumulate / backward / clip / step / zero_grad loop, validation in
eval mode, ``save_pretrained(save_function=, state_dict=)`` checkpoints and the final export."""
import json
import os

import pytest
import torch

from tests.train_script_harness import find_script, make_config, run_script
from tests.test_v1_plumbing_cpu import _fake_ops

SCRIPT = find_script()
needs_script = pytest.mark.skipif(SCRIPT is None, reason="reference training script not available")


def _fake_tokenizer(mp):
    import open_muse_b200.modeling_maskgit_vqgan as V

    def encode(self, pixel_values, return_loss=False):
        g = torch.Generator().manual_seed(int(pixel_values.sum() * 1000) % 100000)
        ids = torch.randint(0, self.num_embeddings, (pixel_values.shape[0], 256), generator=g)
        return None, ids

    def soft(self, pixel_values, temp=1.0, stochastic=False):
        _, ids = encode(self, pixel_values)
        return torch.softmax(torch.randn(ids.shape[0], 256, self.num_embeddings), -1), ids

    mp.setattr(V.MaskGitVQGAN, "encode", encode)
    mp.setattr(V.MaskGitVQGAN, "get_soft_code", soft)


@needs_script
@pytest.mark.parametrize("soft_targets", [False, True])
def test_reference_training_script_runs_unchanged(monkeypatch, tmp_path, soft_targets):
    _fake_ops(monkeypatch)
    _fake_tokenizer(monkeypatch)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    cfg, out = make_config(str(tmp_path), steps=2, batch=3, mixed_precision="no", soft_targets=soft_targets, save_every=2)
    acc = run_script(SCRIPT, cfg)
    steps_logged = [s for v, s in acc.logged if "step_loss" in v]
    assert steps_logged == [1, 2]
    assert any("eval_loss" in v for v, _ in acc.logged)            # validate_model at the end of training
    assert any(k.startswith("grad_norm/") for v, _ in acc.logged for k in v)
    # final export + the step-2 checkpoint written through save_pretrained(save_function=accelerator.save, state_dict=...)
    assert sorted(os.listdir(out))[:2] == ["checkpoint-2", "config.json"] or "pytorch_model.bin" in os.listdir(out)
    assert os.path.exists(os.path.join(out, "pytorch_model.bin")) and os.path.exists(os.path.join(out, "config.yaml"))
    ck = os.path.join(out, "checkpoint-2")
    assert json.load(open(os.path.join(ck, "metadata.json"))) == {"global_step": 2}
    assert os.path.exists(os.path.join(ck, "unwrapped_model", "pytorch_model.bin"))
    cfg_json = json.load(open(os.path.join(out, "config.json")))
    assert cfg_json["_class_name"] == "MaskGitTransformer" and cfg_json["mask_token_id"] == 74


# model.transformer of the reference's configs/imagenet.yaml (the config this script is written for): hidden 768 with 16 heads
# = head_dim 48, vocabulary 2048, 264 positions
IMAGENET_YAML_TRANSFORMER = dict(
    vocab_size=2048, max_position_embeddings=264, hidden_size=768, num_hidden_layers=24, num_attention_heads=16,
    intermediate_size=3072, codebook_size=1024, num_vq_tokens=256, num_classes=1000, initializer_range=0.02,
    norm_type="layernorm", layer_norm_eps=1e-6, use_normformer=True, use_encoder_layernorm=True, use_mlm_layer=True,
    use_mlm_layernorm=True, use_bias=False, hidden_dropout=0.0, attention_dropout=0.0)


@needs_script
def test_reference_training_script_with_its_own_imagenet_yaml_model(monkeypatch, tmp_path):
    """The same unmodified script with the transformer section of the reference's configs/imagenet.yaml (depth cut from 24 to 2
    layers for time): the constructor accepts head_dim 48 and the step loop runs (stand-in kernels; the kernels themselves are
    checked at these widths by tests/test_model_gpu.py::test_head_dim_48_vs_reference_and_oracle)."""
    import yaml

    ref_yaml = os.path.join(os.path.dirname(os.path.dirname(SCRIPT)), "configs", "imagenet.yaml")
    if os.path.exists(ref_yaml):  # the literal above is the reference's, key for key
        ref_tr = yaml.safe_load(open(ref_yaml))["model"]["transformer"]
        ref_tr["layer_norm_eps"] = float(ref_tr["layer_norm_eps"])  # PyYAML reads "1e-6" as a string, OmegaConf as a float
        assert ref_tr == IMAGENET_YAML_TRANSFORMER
    _fake_ops(monkeypatch)
    _fake_tokenizer(monkeypatch)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    cfg, out = make_config(str(tmp_path), steps=2, batch=2, mixed_precision="no",
                           transformer=dict(IMAGENET_YAML_TRANSFORMER, num_hidden_layers=2))
    acc = run_script(SCRIPT, cfg)
    assert [s for v, s in acc.logged if "step_loss" in v] == [1, 2]
    cfg_json = json.load(open(os.path.join(out, "config.json")))
    assert cfg_json["hidden_size"] == 768 and cfg_json["num_attention_heads"] == 16 and cfg_json["mask_token_id"] == 2047


def _lr_sequence(make):
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=0.5)
    sch = make(opt)
    seq = []
    for _ in range(12):
        opt.step()
        sch.step()
        seq.append(sch.get_last_lr()[0])
    return seq


# the named constructors of the reference module with non-default arguments
LR_CASES = [("get_cosine_schedule_with_warmup", dict(num_warmup_steps=2, num_training_steps=10, num_cycles=1.5)),
            ("get_cosine_schedule_with_warmup", dict(num_warmup_steps=2, num_training_steps=10, num_cycles=1)),
            ("get_cosine_with_hard_restarts_schedule_with_warmup", dict(num_warmup_steps=2, num_training_steps=10, num_cycles=3)),
            ("get_polynomial_decay_schedule_with_warmup", dict(num_warmup_steps=2, num_training_steps=10, lr_end=1e-3, power=2.0)),
            ("get_linear_schedule_with_warmup", dict(num_warmup_steps=2, num_training_steps=10)),
            ("get_constant_schedule_with_warmup", dict(num_warmup_steps=2)), ("get_constant_schedule", {})]


def test_lr_schedulers_match_reference():
    """compat muse.lr_schedulers.get_scheduler against the reference's, every schedule name, 12 steps (the reference's
    learning rates are stored in tests/golden/ref_lr_schedulers.json by make_golden.py::make_lr_schedulers)."""
    import sys

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_lr_schedulers.json")) as f:
        ref = json.load(f)
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "open_muse_b200", "compat"))
    try:
        for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
            del sys.modules[k]
        import muse.lr_schedulers as mine
    finally:
        sys.path.pop(0)
    assert list(mine.NAMES) == list(ref["get_scheduler"])
    for name, want in ref["get_scheduler"].items():
        got = _lr_sequence(lambda o: mine.get_scheduler(name, optimizer=o, num_warmup_steps=3, num_training_steps=10))
        assert got == pytest.approx(want, rel=1e-12, abs=1e-15), name
    for fn, kw, want in ref["constructors"]:
        assert _lr_sequence(lambda o: getattr(mine, fn)(o, **kw)) == pytest.approx(want, rel=1e-12, abs=1e-15), fn
    assert [e.value for e in mine.SchedulerType] == ref["scheduler_types"]
    assert set(mine.TYPE_TO_SCHEDULER_FUNCTION) == set(mine.SchedulerType)
    for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
        del sys.modules[k]


@needs_script
@pytest.mark.parametrize("soft_targets", [False, True])
def test_reference_training_script_trains_on_the_numeric_restatements(monkeypatch, tmp_path, soft_targets):
    """The same unmodified script with NUMERIC torch restatements of the kernels (tests/cpu_math_ops.py, precision-recipe
    mode) instead of the shape-checking stand-ins, tokenizer included: images -> MaskGitVQGAN ids / soft codes -> masking ->
    forward + CE -> hand-written backward -> clip -> AdamW.  The loss the script logs is then a real loss: ~log(vocab) at
    the random init and falling."""
    import math

    from tests import cpu_math_ops

    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    steps = 6
    cfg, out = make_config(str(tmp_path), steps=steps, batch=4, mixed_precision="no", soft_targets=soft_targets, save_every=3)
    acc = run_script(SCRIPT, cfg)
    losses = [v["step_loss"] for v, s in acc.logged if "step_loss" in v]
    assert len(losses) == steps and all(math.isfinite(x) for x in losses)
    assert abs(losses[0] - math.log(64 if soft_targets else 75)) < 0.5 and losses[-1] < losses[0], losses
    ev = [v["eval_loss"] for v, s in acc.logged if "eval_loss" in v]
    assert ev and math.isfinite(ev[-1])


@needs_script
def test_reference_offline_ema_script_runs_unchanged(monkeypatch, tmp_path):
    """scripts/compute_offline_ema.py of the reference (load_config / from_pretrained over the checkpoint-N/unwrapped_model
    directories a training run leaves behind, EMAModel.step / copy_to, save_pretrained), unmodified, against the drop-in
    package -- on the checkpoints written by the unmodified training script above.  Host-side only (no kernel is involved)."""
    import runpy
    import sys

    script = os.path.join(os.path.dirname(os.path.dirname(SCRIPT)), "scripts", "compute_offline_ema.py")
    if not os.path.exists(script):
        pytest.skip("reference scripts/ not available (only muse/ and training/ are snapshotted to the GPU box)")
    _fake_ops(monkeypatch)
    _fake_tokenizer(monkeypatch)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    cfg, out = make_config(str(tmp_path), steps=4, batch=2, mixed_precision="no", save_every=2)
    run_script(SCRIPT, cfg)
    assert {"checkpoint-2", "checkpoint-4"} <= set(os.listdir(out))
    compat = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "open_muse_b200", "compat")
    ema_dir = str(tmp_path / "ema")
    saved_argv, saved_path = list(sys.argv), list(sys.path)
    for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
        del sys.modules[k]
    sys.path.insert(0, compat)
    sys.argv = [script, "--checkpoint_dir_path", out, "--ema_save_path", ema_dir, "--ema_decay", "0.5",
                "--checkpoint_interval", "2"]
    try:
        runpy.run_path(script, run_name="__main__")
    finally:
        sys.argv[:], sys.path[:] = saved_argv, saved_path
        for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
            del sys.modules[k]
    from open_muse_b200 import EMAModel, MaskGitTransformer

    got = MaskGitTransformer.from_pretrained(ema_dir).state_dict()
    # the same schedule by hand: shadow = checkpoint-2 weights; steps 1..4, an update on every second one, with the model
    # swapped to checkpoint-2 at step 2 and checkpoint-4 at step 4
    m = MaskGitTransformer.from_pretrained(os.path.join(out, "checkpoint-2", "unwrapped_model"))
    ema = EMAModel(parameters=m.parameters(), decay=0.5, update_every=2)
    for step in range(4):
        if (step + 1) % 2 == 0:
            m = MaskGitTransformer.from_pretrained(os.path.join(out, f"checkpoint-{step + 1}", "unwrapped_model"))
        ema.step(m.parameters())
    ema.copy_to(m.parameters())
    for k, v in m.state_dict().items():
        assert torch.equal(got[k], v), k


@needs_script
def test_reference_training_script_resumes_from_its_checkpoint(monkeypatch, tmp_path):
    """Checkpoint / resume of the unmodified script (train_maskgit_imagenet.py:329-355): a 4-step run that saved at step 2
    is resumed with ``experiment.resume_from_checkpoint=latest`` for two more steps -- model weights, AdamW moments and the
    LR schedule come back from checkpoint-2 (the step counter from the directory name), and the run ends with the same
    checkpoint layout, AdamW's own step counter continuing at 3.  Runs on the numeric kernel restatements."""
    from tests import cpu_math_ops

    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    # run A: 2 steps, checkpoint at 2
    cfg, out = make_config(str(tmp_path), steps=2, batch=3, mixed_precision="no", save_every=2)
    acc = run_script(SCRIPT, cfg)
    assert [s for v, s in acc.logged if "step_loss" in v] == [1, 2]
    sd2 = torch.load(os.path.join(out, "checkpoint-2", "unwrapped_model", "pytorch_model.bin"))
    # run B: same config, resume, train to step 4
    acc = run_script(SCRIPT, cfg, extra_cli=("experiment.resume_from_checkpoint=latest", "training.max_train_steps=4"))
    steps = [s for v, s in acc.logged if "step_loss" in v]
    assert steps == [3, 4], steps
    assert json.load(open(os.path.join(out, "checkpoint-4", "metadata.json"))) == {"global_step": 4}
    sd4 = torch.load(os.path.join(out, "checkpoint-4", "unwrapped_model", "pytorch_model.bin"))
    w = "transformer_layers.0.ffn.wi_0.weight"
    assert not torch.equal(sd2[w], sd4[w])
    opt = torch.load(os.path.join(out, "checkpoint-4", "optimizer.bin"))
    assert int(next(iter(opt["state"].values()))["step"]) == 4  # AdamW's own step counter continued from the loaded state


@needs_script
def test_reference_benchmark_models_script_runs_unchanged(monkeypatch, tmp_path, capsys):
    """scripts/benchmark_models.py of the reference, unmodified (load_config / from_config, text-conditional generate2 in
    fp32, after ``model.half()`` and after enable_xformers_memory_efficient_attention(), timed with torch.utils.benchmark),
    against the drop-in package on the numeric kernel restatements: the calls it makes exist and run end to end."""
    import runpy
    import sys

    script = os.path.join(os.path.dirname(os.path.dirname(SCRIPT)), "scripts", "benchmark_models.py")
    if not os.path.exists(script):
        pytest.skip("reference scripts/ not available")
    from open_muse_b200 import MaskGitTransformer
    from tests import cpu_math_ops

    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setattr(MaskGitTransformer, "device", property(lambda self: torch.device("cpu")), raising=False)
    monkeypatch.setenv("MUSE_B200_GENERATE_GRAPH", "0")
    cfg_dir = str(tmp_path / "cfg")
    MaskGitTransformer(vocab_size=72, hidden_size=64, num_hidden_layers=1, num_attention_heads=1, intermediate_size=128,
                       hidden_dropout=0.0, attention_dropout=0.0, max_position_embeddings=16, codebook_size=64, num_vq_tokens=16,
                       add_cross_attention=True, encoder_hidden_size=32, use_codebook_size_for_output=True).save_config(cfg_dir)
    compat = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "open_muse_b200", "compat")
    saved_argv, saved_path = list(sys.argv), list(sys.path)
    for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
        del sys.modules[k]
    sys.path.insert(0, compat)
    sys.argv = [script, "--config_path", cfg_dir, "--batch_size", "2", "--text_length", "5", "--time_steps", "2", "--device", "cpu"]
    try:
        runpy.run_path(script, run_name="__main__")
    finally:
        sys.argv[:], sys.path[:] = saved_argv, saved_path
        for k in [k for k in sys.modules if k == "muse" or k.startswith("muse.")]:
            del sys.modules[k]
    out = capsys.readouterr().out
    assert "Vanilla attention in FP32" in out and "Efficient attention in FP16" in out


@needs_script
def test_reference_training_script_with_gradient_accumulation(monkeypatch, tmp_path):
    """training.gradient_accumulation_steps = 2: the script's ``accelerator.accumulate(model)`` windows -- gradients of two
    micro-batches add up in the parameters' .grad (each per-layer Function hands its gradients to autograd's accumulation) and
    the optimizer / scheduler act once per window."""
    import math

    from tests import cpu_math_ops

    cpu_math_ops.install(monkeypatch, exact=False)
    monkeypatch.setenv("ACCELERATE_USE_CPU", "1")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    cfg, out = make_config(str(tmp_path), steps=3, batch=2, mixed_precision="no", save_every=3)
    acc = run_script(SCRIPT, cfg, extra_cli=("training.gradient_accumulation_steps=2",))
    losses = [v["step_loss"] for v, s in acc.logged if "step_loss" in v]
    assert [s for v, s in acc.logged if "step_loss" in v] == [1, 2, 3] and all(math.isfinite(x) for x in losses)
    opt = torch.load(os.path.join(out, "checkpoint-3", "optimizer.bin"))
    assert int(next(iter(opt["state"].values()))["step"]) == 3  # six micro-batches, three optimizer steps
